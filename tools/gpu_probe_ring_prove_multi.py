#!/usr/bin/env python
"""GPU probe: Ring VRF proving over several rings in one call (dr_ring_prove_multi); writes its results as JSON to $PROBE_OUT (default:
probe_ring_prove_multi.json in the temporary directory).

  python tools/gpu_probe_ring_prove_multi.py [PARENT_LIB]

- no regression: dr_ring_prove_batch of 4096 proofs at ring 1023 with the bench's default table (16-bit windows over GLV halves), with
  this tree's library and (when PARENT_LIB, a build of the parent commit, is given) that library: one process per library and run,
  the processes alternated, each timing REPS calls after a warm-up call;
- gain: 4096 proofs at ring 1023 over K = 1, 8, 64 rings as one dr_ring_prove_multi call against K dr_ring_prove_batch calls of
  4096 / K proofs each, every proof of the multi call checked against the loop's;
- memory: device bytes 64 rings of 1023 keys hold beyond the shared window table (free-memory delta after a trim).
Times are device times (CUDA events on the context stream around the whole call) and host wall-clock times after a synchronise.
The card's name, power limit and maximum SM clock are read in the same run."""
import ctypes
import json
import os
import random
import subprocess
import sys
import tempfile
import time
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dot_ring_b200 import _native  # noqa: E402
from dot_ring_b200.srs import read_srs_file  # noqa: E402
from oracle import bandersnatch as bs  # noqa: E402
from oracle import fr, ring_proof as rp  # noqa: E402
from oracle import transcript as otr  # noqa: E402
from tests.helpers import bench_ring_keys, le64, seed  # noqa: E402
from tests.ring_fixtures import native_ring  # noqa: E402

REPS = int(os.environ.get("REPS", "8"))
N = 4096
out = {"reps": REPS, "table": "16-bit windows over GLV halves (bench.py default)"}
try:
    out["nvidia_smi"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                                       timeout=60).stdout.strip()
except Exception as e:  # noqa: BLE001
    out["nvidia_smi"] = f"unavailable: {e}"
print(out["nvidia_smi"], flush=True)


class _Tolerant:
    """ctypes library view for _declare on a parent build: entry points it lacks (dr_ring_prove_multi) are skipped."""

    def __init__(self, lib):
        self.lib = lib

    def __getattr__(self, name):
        try:
            return getattr(self.lib, name)
        except AttributeError:
            return types.SimpleNamespace()


AB_ONLY = len(sys.argv) > 2 and sys.argv[1] == "--ab"
if AB_ONLY:  # child: dr_ring_prove_batch timings with the library at argv[2] (a build of this or of the parent commit)
    lib = _native.Library.__new__(_native.Library)
    lib.path = sys.argv[2]
    lib.lib = ctypes.CDLL(sys.argv[2])
    _native.Library._declare(types.SimpleNamespace(lib=_Tolerant(lib.lib)))
    assert lib.lib.dr_is_cuda_build()
else:
    lib = _native.Library()
ctx = _native.Context(0, lib)
out["device"] = ctx.device_info()
params = rp.Params.from_ring_size(1023)
pk, sk, base_keys = bench_ring_keys(1023)


def ring_keys(r: int):
    keys = list(base_keys)
    if r:
        keys[1000] = otr.secret_from_seed(bs.SHA512, seed("probe-ring", r))[0]
    return keys


def bench_srs(c):
    raw = read_srs_file(None, None)
    return _native.NativeSrs(c, raw.g1_be96, raw.g2_be192, 16, 0, glv=True)


def timed(c, fn):
    c.sync()
    t0 = time.perf_counter()
    c.timer_start()
    res = fn()
    ms = c.timer_stop()
    return res, ms, (time.perf_counter() - t0) * 1e3


def stats(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1], "all": xs}


def batch(r: int, cnt: int):
    rng = random.Random(r)
    al = [b"probe-input-%d-" % r + le64(j) for j in range(cnt)]
    ad = [b"probe-ad-%d-" % r + le64(j) for j in range(cnt)]
    return al, ad, [rng.randrange(fr.R) for _ in range(12 * cnt)]


if AB_ONLY:  # ---- no regression, one library: dr_ring_prove_batch of 4096 proofs
    srs = bench_srs(ctx)
    ring = native_ring(srs, ring_keys(0), params)
    al, ad, zk = batch(0, N)
    dev_ms, wall_ms, first = [], [], None
    for rep in range(REPS + 1):
        (pr, st), dev, wall = timed(ctx, lambda: ring.prove_batch(al, ad, [sk] * N, [3] * N, zk_rows=zk))
        assert not any(st)
        first = first or pr[0] + pr[-1]
        if rep:  # rep 0 warms up
            dev_ms.append(dev)
            wall_ms.append(wall)
    print("AB_RESULT " + json.dumps({"device_ms": dev_ms, "wall_ms": wall_ms, "first_last_proof": first.hex()}), flush=True)
    sys.exit(0)

# ---- no regression: dr_ring_prove_batch, this tree's library and the parent's, alternated processes (before this process builds
# its own table: the 161 GB table fits the card once) ----------------------------------------------------------------------------
runs = {"branch": str(_native.DEFAULT_LIBRARY)}
if len(sys.argv) > 1:
    runs["parent"] = sys.argv[1]
ab = {k: {"device_ms": [], "wall_ms": [], "first_last_proof": set()} for k in runs}
for rep in range(int(os.environ.get("AB_PROCESSES", "4"))):
    for k in (list(runs) if rep % 2 == 0 else list(runs)[::-1]):
        proc = subprocess.run([sys.executable, os.path.abspath(__file__), "--ab", runs[k]], capture_output=True, text=True, timeout=600)
        line = [x for x in proc.stdout.splitlines() if x.startswith("AB_RESULT ")]
        assert proc.returncode == 0 and line, (k, proc.stdout[-2000:], proc.stderr[-2000:])
        d = json.loads(line[0][len("AB_RESULT "):])
        ab[k]["device_ms"] += d["device_ms"]
        ab[k]["wall_ms"] += d["wall_ms"]
        ab[k]["first_last_proof"].add(d["first_last_proof"])
        print(k, rep, stats(d["device_ms"])["median"], flush=True)
out["prove_batch_4096_ring1023"] = {k: {"device_ms": stats(v["device_ms"]), "wall_ms": stats(v["wall_ms"])} for k, v in ab.items()}
out["same_proofs_as_parent"] = len(set().union(*[v["first_last_proof"] for v in ab.values()])) == 1
print({k: out["prove_batch_4096_ring1023"][k]["device_ms"]["median"] for k in runs}, "same proofs:", out["same_proofs_as_parent"], flush=True)

# ---- memory: 64 rings beyond the shared table ---------------------------------------------------------------------------------
srs = bench_srs(ctx)
rings = [native_ring(srs, ring_keys(0), params)]
al, ad, zk = batch(0, 8)
rings[0].prove_batch(al, ad, [sk] * 8, [3] * 8, zk_rows=zk)  # the Lagrange table of N = 2048 is built at the first proof
ctx.trim()
ctx.sync()
free0 = ctx.device_info()["free_bytes"]
rings += [native_ring(srs, ring_keys(r), params) for r in range(1, 64)]
ctx.trim()
ctx.sync()
free1 = ctx.device_info()["free_bytes"]
out["ring_device_bytes"] = {"63 rings of 1023 keys (free-memory delta)": free0 - free1, "per ring": (free0 - free1) / 63}
print(out["ring_device_bytes"], flush=True)

# ---- gain: one multi call vs K dr_ring_prove_batch calls ----------------------------------------------------------------------
gain = {}
for K in (1, 8, 64):
    per = N // K
    members = list(range(K))
    parts = [batch(r, per) for r in members]
    al = [a for p in parts for a in p[0]]
    ad = [d for p in parts for d in p[1]]
    zk = [z for p in parts for z in p[2]]
    index = [r for r in members for _ in range(per)]
    multi_dev, multi_wall, loop_dev, loop_wall = [], [], [], []
    for rep in range(REPS + 1):
        (pr, st), dev, wall = timed(ctx, lambda: _native.NativeRing.prove_multi([rings[r] for r in members], index, al, ad, [sk] * N, [3] * N, zk))
        assert not any(st), K
        if rep:
            multi_dev.append(dev)
            multi_wall.append(wall)

        def loop():
            return [rings[r].prove_batch(al[r * per : (r + 1) * per], ad[r * per : (r + 1) * per], [sk] * per, [3] * per, zk[12 * r * per : 12 * (r + 1) * per])
                    for r in members]

        res, dev, wall = timed(ctx, loop)
        assert [p for proofs, _ in res for p in proofs] == pr, K
        if rep:
            loop_dev.append(dev)
            loop_wall.append(wall)
    gain[f"K{K}"] = {"multi_device_ms": stats(multi_dev), "multi_wall_ms": stats(multi_wall), "loop_device_ms": stats(loop_dev), "loop_wall_ms": stats(loop_wall)}
    print(K, gain[f"K{K}"]["multi_device_ms"]["median"], gain[f"K{K}"]["loop_device_ms"]["median"], flush=True)
out["multi_vs_loop_4096"] = gain
path = os.environ.get("PROBE_OUT") or os.path.join(tempfile.gettempdir(), "probe_ring_prove_multi.json")
os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
with open(path, "w") as f:
    json.dump(out, f, indent=1)
print("wrote", path, flush=True)
print(json.dumps({k: v for k, v in out.items() if k == "nvidia_smi"}))
