#!/usr/bin/env python
"""GPU probe: ring roots from keys without a Ring or the prover's window table (RingRoot.from_keys / from_key_sets / update); writes
its results as JSON to $PROBE_OUT (default: probe_ring_roots.json in the temporary directory).

  python tools/gpu_probe_ring_roots.py

- from_keys of 1023 keys at N = 2048 on a fresh engine: the first call (which builds the small root table) and the steady state; the
  table's bytes and the drop in free device memory;
- for comparison, Ring(keys) + RingRoot.from_ring on an engine whose default window table is built, and that table's build time;
- 64 rings of 1023 keys in one from_key_sets call against 64 from_keys calls;
- updates of 1, 16 and 256 rows at N = 2048;
- from_keys of 65279 keys at N = 65536 over a 65536-point synthetic SRS.
Device times are CUDA events on the context stream around the whole call; wall times are host clocks around a call that ends in a
synchronise.  The card's name and power limit are read in the same run."""
import json
import os
import random
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dot_ring_b200 as api  # noqa: E402
from dot_ring_b200 import engine as engine_mod  # noqa: E402
from dot_ring_b200.srs import SrsBytes, read_srs_file  # noqa: E402
from oracle import bandersnatch as bs  # noqa: E402
from oracle import transcript as otr  # noqa: E402
from tests.helpers import bench_ring_keys, seed  # noqa: E402
from tests.msm_cases import TAU  # noqa: E402

REPS = int(os.environ.get("REPS", "10"))
out = {"reps": REPS}
try:
    out["nvidia_smi"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                                       timeout=60).stdout.strip()
except Exception as e:  # noqa: BLE001
    out["nvidia_smi"] = f"unavailable: {e}"
print(out["nvidia_smi"], flush=True)


def timed(eng, fn):
    """(result, device ms, wall ms) of fn() on eng's context stream."""
    eng.ctx.sync()
    t0 = time.perf_counter()
    eng.ctx.timer_start()
    res = fn()
    dev = eng.ctx.timer_stop()
    return res, dev, (time.perf_counter() - t0) * 1e3


def repeat(eng, fn, reps=REPS):
    dev, wall = [], []
    for _ in range(reps):
        _, d, w = timed(eng, fn)
        dev.append(d)
        wall.append(w)
    return {"device_ms": stats(dev), "wall_ms": stats(wall)}


def stats(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1]}


params = api.RingProofParams.from_ring_size(1023)
assert params.domain_size == 2048
_, _, keys = bench_ring_keys(1023)


def ring_keys(r: int):
    k = list(keys)
    if r:
        k[1000] = otr.secret_from_seed(bs.SHA512, seed("probe-root-ring", r))[0]
    return k


# ---- from_keys on a fresh engine -------------------------------------------------------------------------------------------
eng = engine_mod.Engine(0)
out["device"] = eng.ctx.device_info()
free0 = eng.ctx.device_info()["free_bytes"]
root, dev, wall = timed(eng, lambda: api.RingRoot.from_keys(keys, params, eng))
free1 = eng.ctx.device_info()["free_bytes"]
out["from_keys_1023_n2048"] = {
    "first_call": {"device_ms": dev, "wall_ms": wall},
    "steady": repeat(eng, lambda: api.RingRoot.from_keys(keys, params, eng)),
    "root_table_bytes": eng.root_srs(2048).table_bytes,
    "free_device_bytes_drop": free0 - free1,
    "window_table_built": eng._srs is not None,
}
print("from_keys", out["from_keys_1023_n2048"], flush=True)

# ---- 64 rings: one call against 64 calls -------------------------------------------------------------------------------------
sets = [ring_keys(r) for r in range(64)]
one = api.RingRoot.from_key_sets(sets, params, eng)
assert [r.fixed_commitments() for r in one] == [api.RingRoot.from_keys(s, params, eng).fixed_commitments() for s in sets]
out["rings64_1023_n2048"] = {
    "one_call": repeat(eng, lambda: api.RingRoot.from_key_sets(sets, params, eng), max(3, REPS // 3)),
    "64_calls": repeat(eng, lambda: [api.RingRoot.from_keys(s, params, eng) for s in sets], max(3, REPS // 3)),
}
print("64 rings", out["rings64_1023_n2048"], flush=True)

# ---- updates -----------------------------------------------------------------------------------------------------------------
rng = random.Random(1)
fresh = eng.ctx.te_mul([bs.point_to_string(bs.GENERATOR)], [rng.randrange(1, bs.N) for _ in range(256)])
updates = {}
for n in (1, 16, 256):
    rows = rng.sample(range(1023), n)
    new = fresh[:n]
    changed = list(keys)
    for r, k in zip(rows, new):
        changed[r] = k
    upd = root.update(rows, new, [keys[r] for r in rows])
    assert upd.fixed_commitments() == api.RingRoot.from_keys(changed, params, eng).fixed_commitments()
    updates[str(n)] = repeat(eng, lambda: root.update(rows, new, [keys[r] for r in rows]))
out["update_n2048"] = updates
print("updates", updates, flush=True)

# ---- the prover's route on an engine whose default table is built --------------------------------------------------------------
ref = engine_mod.Engine(0)
t0 = time.perf_counter()
ref.srs
ref.ctx.sync()
out["default_table"] = {"build_s": time.perf_counter() - t0, "bytes": ref.srs.table_bytes, "geometry": ref.srs.geometry}


def via_ring():
    ring = api.Ring(keys, params, ref)
    r = api.RingRoot.from_ring(ring)
    ring.native.close()
    return r


r, dev, wall = timed(ref, via_ring)
assert r.fixed_commitments() == root.fixed_commitments()
out["ring_plus_from_ring_1023_n2048"] = {"first_call": {"device_ms": dev, "wall_ms": wall}, "steady": repeat(ref, via_ring)}
print("default table", out["default_table"], "ring route", out["ring_plus_from_ring_1023_n2048"], flush=True)
ref.close()
eng.close()

# ---- N = 65536 over a synthetic SRS ------------------------------------------------------------------------------------------
big_params = api.RingProofParams(domain_size=65536, max_domain_size=65536)
g2 = read_srs_file(None, 1).g2_be192  # not used by the root functions
tmp = engine_mod.Engine(0, srs_points=1)
g1 = tmp.ctx.g1_synthetic_srs(TAU, 0, 65536)
tmp.close()
big = engine_mod.Engine(0, srs=SrsBytes(g1, g2))
big_keys = big.ctx.te_mul([bs.point_to_string(bs.GENERATOR)], [rng.randrange(1, bs.N) for _ in range(big_params.max_ring_size)])
free0 = big.ctx.device_info()["free_bytes"]
_, dev, wall = timed(big, lambda: api.RingRoot.from_keys(big_keys, big_params, big))
free1 = big.ctx.device_info()["free_bytes"]
out["from_keys_n65536"] = {
    "keys": len(big_keys),
    "first_call": {"device_ms": dev, "wall_ms": wall},
    "steady": repeat(big, lambda: api.RingRoot.from_keys(big_keys, big_params, big), max(3, REPS // 3)),
    "root_table_bytes": big.root_srs(65536).table_bytes,
    "free_device_bytes_drop": free0 - free1,
}
print("n65536", out["from_keys_n65536"], flush=True)
big.close()

path = os.environ.get("PROBE_OUT") or os.path.join(tempfile.gettempdir(), "probe_ring_roots.json")
with open(path, "w") as f:
    json.dump(out, f, indent=1, default=str)
print("wrote", path)
