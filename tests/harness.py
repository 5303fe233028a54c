"""Differential-testing harness.

A *script* is a deterministic list of steps (map commands and batch runs).
``run_script`` executes it on a backend — the reference oracle, the port
oracle, or the GPU dataplane — and returns everything observable: per-run
verdicts / rewritten frames / lengths / priorities, return codes of map
commands, final counters, table contents and event streams.  ``compare``
asserts two result sets are bit-identical (compiler padding masked).
"""
from __future__ import annotations

import hashlib

import numpy as np

from bng_b200 import layouts as L
from bng_b200.layouts import as_bytes

STATS_MAPS = ("antispoof_stats", "qos_stats_map", "nat_stats_map", "stats_map")
EVENT_MAPS = ("spoof_events", "nat_log_rb")
TABLES = ("subscriber_bindings", "qos_egress", "qos_ingress", "nat_sessions", "nat_reverse", "eim_table",
          "subscriber_nat", "hairpin_ips", "alg_ports", "subscriber_pools", "vlan_subscriber_pools", "ip_pools",
          "circuit_id_map", "circuit_id_subscribers", "allowed_ranges_v4", "antispoof_config", "nat_config_map",
          "server_config", "nat_pool")


def mask_padding(name: str, vals: np.ndarray) -> np.ndarray:
    v = vals.copy()
    for off, ln in L.PADDING.get(name, ()):
        if v.shape[1] >= off + ln:
            v[:, off:off + ln] = 0
    return v


# ---------------------------------------------------------------------------
# script construction
# ---------------------------------------------------------------------------
class Script:
    def __init__(self, name: str):
        self.name = name
        self.steps = []

    def update(self, m, keys, vals, flags=0):
        k, v = as_bytes(np.asarray(keys)), as_bytes(np.asarray(vals))
        if k.shape[0] != v.shape[0]:  # single key given as bytes
            k = k.reshape(1, -1)
            v = v.reshape(1, -1)
        self.steps.append(("update", m, k.copy(), v.copy(), flags))
        return self

    def update1(self, m, key, val, flags=0):
        k = as_bytes(np.asarray(key)).reshape(1, -1)
        v = as_bytes(np.asarray(val)).reshape(1, -1)
        self.steps.append(("update", m, k, v, flags))
        return self

    def delete(self, m, key):
        self.steps.append(("delete", m, as_bytes(np.asarray(key)).reshape(-1).copy()))
        return self

    def lookup(self, m, key):
        self.steps.append(("lookup", m, as_bytes(np.asarray(key)).reshape(-1).copy()))
        return self

    def run(self, prog, arena, lens, now_ns, off16=None, stride=0, priority=None, now_v=None):
        """now_v: bpf_ktime_get_ns() per frame (u64[n], non-decreasing) instead of one value for the batch."""
        if off16 is None and stride == 0:
            stride = 64
        self.steps.append(("run", prog, arena.copy(), lens.astype(np.uint32).copy(), int(now_ns),
                           None if off16 is None else off16.astype(np.uint32).copy(), int(stride),
                           None if priority is None else priority.astype(np.uint32).copy(),
                           None if now_v is None else np.ascontiguousarray(now_v, dtype=np.uint64).copy()))
        return self

    def drain(self):
        """Drain both event rings at this point (frees nat_log_rb space)."""
        self.steps.append(("drain",))
        return self

    def run_from(self, prog, fn):
        """A run whose inputs are derived from earlier results: fn(results) ->
        dict(arena=, lens=, now_ns=, [off16=], [stride=], [priority=])."""
        self.steps.append(("run_from", prog, fn))
        return self


# ---------------------------------------------------------------------------
# backends
# ---------------------------------------------------------------------------
class OracleBackend:
    def __init__(self, kind: str):
        from oracle.pyoracle import Oracle
        self.o = Oracle(kind)
        self.kind = kind

    def close(self):
        self.o.free_arenas()

    def update(self, m, k, v, flags):
        return self.o.update_batch(m, k, v, flags)

    def delete(self, m, k):
        return self.o.delete(m, k)

    def lookup(self, m, k):
        return self.o.lookup(m, k)

    def run(self, prog, arena, lens, now, off16, stride, prio, now_v=None):
        oa = self.o.arena(len(arena) + 64)
        oa[:len(arena)] = arena
        v = self.o.run(prog, oa, lens, now, off16=off16, stride=stride, priority=prio, now_v=now_v)
        arena[:] = oa[:len(arena)]
        self.o.free_arenas()
        return v

    def stats(self, m):
        return self.o.lookup(m, np.zeros(4, np.uint8)).view("<u8").copy()

    def dump(self, m):
        return self.o.dump(m)

    def drain(self, m):
        return self.o.drain(m)

    def health(self):
        return {}


class GpuBackend:
    def __init__(self, dp=None, pinned=False, **opts):
        self.pinned = pinned
        if dp is None:
            from bng_b200 import Dataplane
            opts.setdefault("max_subscribers", 1 << 14)
            opts.setdefault("max_nat_sessions", 1 << 16)
            opts.setdefault("max_eim_mappings", 1 << 16)
            opts.setdefault("max_batch", 1 << 16)
            opts.setdefault("event_capacity", 1 << 16)
            dp = Dataplane(**opts)
        self.dp = dp
        self.kind = "gpu"

    def close(self):
        self.dp.close()

    def update(self, m, k, v, flags):
        return self.dp.update_batch(m, k, v, flags)

    def delete(self, m, k):
        return self.dp.delete(m, k)

    def lookup(self, m, k):
        return self.dp.lookup(m, k)

    def run(self, prog, arena, lens, now, off16, stride, prio, now_v=None):
        if not getattr(self, "pinned", False):
            return self.dp.run(prog, arena, lens, now, off16=off16, stride=stride, priority=prio, now_v=now_v)
        # pinned host buffers: exercises the zero-copy gather/scatter path of BNG_MEM_HOST
        import torch
        from bng_b200 import MEM_HOST
        if self.pinned == "abi":  # the arena comes from bng_host_alloc() (huge-page backed, registered)
            import ctypes
            from bng_b200.dataplane import load_library
            lib = load_library()
            p = lib.bng_host_alloc(arena.nbytes + 64)
            assert p, "bng_host_alloc failed"
            try:
                view = np.ctypeslib.as_array((ctypes.c_uint8 * arena.nbytes).from_address(p))
                view[:] = arena
                tl = torch.from_numpy(lens.view(np.int32).copy()).pin_memory()
                to = None if off16 is None else torch.from_numpy(off16.view(np.int32).copy()).pin_memory()
                tp = None if prio is None else torch.from_numpy(prio.view(np.int32).copy()).pin_memory()
                tv = torch.zeros(len(lens), dtype=torch.uint8).pin_memory()
                tn = None if now_v is None else torch.from_numpy(now_v.view(np.int64).copy()).pin_memory()
                self.dp.run(prog, int(p), tl, now, off16=to, stride=stride, priority=tp, verdict=tv, mem=MEM_HOST,
                            arena_bytes=arena.nbytes, now_v=tn)
                arena[:] = view
            finally:
                lib.bng_host_free(p)
            lens[:] = tl.numpy().view(np.uint32)
            if prio is not None:
                prio[:] = tp.numpy().view(np.uint32)
            return tv.numpy().copy()
        ta = torch.from_numpy(arena.copy()).pin_memory()
        tl = torch.from_numpy(lens.view(np.int32).copy()).pin_memory()
        to = None if off16 is None else torch.from_numpy(off16.view(np.int32).copy()).pin_memory()
        tp = None if prio is None else torch.from_numpy(prio.view(np.int32).copy()).pin_memory()
        tv = torch.zeros(len(lens), dtype=torch.uint8).pin_memory()
        tn = None if now_v is None else torch.from_numpy(now_v.view(np.int64).copy()).pin_memory()
        self.dp.run(prog, ta, tl, now, off16=to, stride=stride, priority=tp, verdict=tv, mem=MEM_HOST,
                    arena_bytes=arena.nbytes, now_v=tn)
        arena[:] = ta.numpy()
        lens[:] = tl.numpy().view(np.uint32)
        if prio is not None:
            prio[:] = tp.numpy().view(np.uint32)
        return tv.numpy().copy()

    def stats(self, m):
        return self.dp.stats(m)

    def dump(self, m):
        return self.dp.dump(m)

    def drain(self, m):
        return self.dp.drain(m)

    def health(self):
        return {"lru_overflow": self.dp.lru_overflow, "events_lost": self.dp.events_lost}


# ---------------------------------------------------------------------------
# execution and comparison
# ---------------------------------------------------------------------------
def run_script(be, script: Script, tables=TABLES) -> dict:
    res = {}
    events = {m: [] for m in EVENT_MAPS}
    for si, st in enumerate(script.steps):
        tag = f"s{si:03d}"
        if st[0] == "update":
            res[tag + "_rc"] = np.array([be.update(st[1], st[2], st[3], st[4])], dtype=np.int64)
        elif st[0] == "delete":
            res[tag + "_rc"] = np.array([be.delete(st[1], st[2])], dtype=np.int64)
        elif st[0] == "lookup":
            v = be.lookup(st[1], st[2])
            res[tag + "_found"] = np.array([v is not None], dtype=np.int64)
            if v is not None:
                res[tag + "_val"] = mask_padding(st[1], v[None])[0]
        elif st[0] in ("run", "run_from"):
            if st[0] == "run_from":
                d = st[2](res)
                prog, arena, lens, now = st[1], d["arena"], d["lens"].astype(np.uint32), int(d["now_ns"])
                off16, stride, prio, now_v = d.get("off16"), int(d.get("stride", 0)), d.get("priority"), d.get("now_v")
            else:
                _, prog, arena, lens, now, off16, stride, prio, now_v = st
            a, l = arena.copy(), lens.copy()
            p = None if prio is None else prio.copy()
            v = be.run(prog, a, l, now, off16, stride, p, now_v) if now_v is not None else be.run(prog, a, l, now, off16, stride, p)
            res[tag + "_verdict"] = np.asarray(v).copy()
            res[tag + "_frames"] = a
            res[tag + "_len"] = l
            if p is not None:
                res[tag + "_prio"] = p
        elif st[0] == "drain":
            for m in EVENT_MAPS:
                events[m].append(be.drain(m))
    for m in EVENT_MAPS:
        events[m].append(be.drain(m))
        ev = [e for e in events[m] if e.shape[0]]
        if ev:
            res["ev_" + m] = mask_padding(m, np.concatenate(ev, axis=0))
        else:
            res["ev_" + m] = np.zeros((0, 1), np.uint8)
    for m in STATS_MAPS:
        res["st_" + m] = be.stats(m)
    for m in tables:
        k, v = be.dump(m)
        res["tk_" + m] = k
        res["tv_" + m] = mask_padding(m, v) if v.shape[0] else v
    for k, v in be.health().items():
        assert v == 0, f"{script.name}: backend health counter {k} = {v}"
    return res


def diff_keys(a: dict, b: dict) -> list:
    """Every result key on which two result sets differ, as (key, description) pairs."""
    out = []
    for k in sorted(set(a.keys()) ^ set(b.keys())):
        out.append((k, "present on one side only"))
    for k in sorted(set(a.keys()) & set(b.keys())):
        x, y = np.asarray(a[k]), np.asarray(b[k])
        if x.shape[0] == 0 and y.shape[0] == 0:
            continue
        if x.shape != y.shape:
            out.append((k, f"shape {x.shape} vs {y.shape}"))
        elif not np.array_equal(x, y):
            d = np.argwhere(x != y)
            out.append((k, f"{len(d)} elements differ, first at {d[0].tolist()}: {x[tuple(d[0])]} vs {y[tuple(d[0])]}"))
    return out


def compare(a: dict, b: dict, what: str = ""):
    """Asserts bit-identity of two result sets; the failure message lists EVERY differing key (verdicts, frames,
    counters, table dumps, event streams), not just the first in sort order."""
    diffs = diff_keys(a, b)
    if diffs:
        lines = "\n".join(f"  {k}: {msg}" for k, msg in diffs[:40])
        raise AssertionError(f"{what}: {len(diffs)} result keys differ\n{lines}")


def save_golden(path: str, res: dict):
    np.savez_compressed(path, **res)


def load_golden(path: str) -> dict:
    with np.load(path) as z:
        return {k: z[k] for k in z.files}


def fingerprint(res: dict) -> dict:
    """Per result key: the array's shape and the SHA-256 of its bytes (first 64 bits), or "empty" for an array with
    no rows, as diff_keys treats those.  Lets a result set too large to store be pinned bit for bit."""
    out = {}
    for k, v in res.items():
        a = np.ascontiguousarray(v)
        if a.shape[0] == 0:
            out[k] = "empty"
        else:
            out[k] = "x".join(map(str, a.shape)) + ":" + hashlib.sha256(a.tobytes()).hexdigest()[:16]
    return out


def compare_fingerprint(want: dict, res: dict, what: str = ""):
    """compare() against a stored fingerprint(): lists every result key whose shape or bytes differ."""
    got = fingerprint(res)
    diffs = [(k, "present on one side only") for k in sorted(set(want) ^ set(got))]
    diffs += [(k, f"{want[k]} vs {got[k]}") for k in sorted(set(want) & set(got)) if want[k] != got[k]]
    if diffs:
        lines = "\n".join(f"  {k}: {msg}" for k, msg in diffs[:40])
        raise AssertionError(f"{what}: {len(diffs)} result keys differ (shape:sha256)\n{lines}")
