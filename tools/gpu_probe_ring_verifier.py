#!/usr/bin/env python
"""GPU probe: keyless, multi-ring Ring VRF verification (dr_ring_verify_multi); writes its results as JSON to $PROBE_OUT (default:
probe_ring_verifier.json in the temporary directory).

  python tools/gpu_probe_ring_verifier.py [PARENT_LIB]

- no regression: 4096 proofs at ring 1023 through dr_ring_verify_batch per item, aggregated and aggregated by the two-MSM route, with
  this tree's library and (when PARENT_LIB, a build of the parent commit, is given) that library: one process per library and run
  (two builds of the library do not share a process), the processes alternated, each timing every mode REPS times after a warm-up;
- gain: 4096 proofs over K = 1, 8, 64 rings as one dr_ring_verify_multi call against K dr_ring_verify_batch calls, both modes;
- verifier cost: dr_ring_verifier_create time and device memory against dr_srs_load (window table) + dr_ring_create.
Times are device times (CUDA events on the context stream around the whole call) and host wall-clock times after a synchronise."""
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
from oracle import bandersnatch as bs  # noqa: E402
from oracle import fr, ring_proof as rp  # noqa: E402
from oracle import transcript as otr  # noqa: E402
from tests.helpers import bench_ring_keys, le64, seed  # noqa: E402
from tests.ring_fixtures import native_ring, native_srs  # noqa: E402
from tests.ring_verifier_cases import make_verifier  # noqa: E402

REPS = int(os.environ.get("REPS", "5"))
WINDOW_BITS = int(os.environ.get("DR_WINDOW_BITS", "8"))
N = 4096
out = {"reps": REPS, "window_bits": WINDOW_BITS}
try:
    out["nvidia_smi"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                                       timeout=60).stdout.strip()
except Exception as e:  # noqa: BLE001
    out["nvidia_smi"] = f"unavailable: {e}"
print(out["nvidia_smi"], flush=True)


class _Tolerant:
    """ctypes library view for _declare on a parent build: entry points it lacks (dr_ring_verifier_*, dr_ring_verify_multi) are skipped."""

    def __init__(self, lib):
        self.lib = lib

    def __getattr__(self, name):
        try:
            return getattr(self.lib, name)
        except AttributeError:
            return types.SimpleNamespace()


AB_ONLY = len(sys.argv) > 2 and sys.argv[1] == "--ab"
if AB_ONLY:  # child: dr_ring_verify_batch timings with the library at argv[2] (a build of this or of the parent commit)
    lib = _native.Library.__new__(_native.Library)
    lib.path = sys.argv[2]
    lib.lib = ctypes.CDLL(sys.argv[2])
    for name in ("dr_ctx_create", "dr_ctx_destroy", "dr_ctx_sync", "dr_ctx_timer_start", "dr_ctx_timer_stop", "dr_srs_load", "dr_srs_destroy", "dr_ring_create",
                 "dr_ring_destroy", "dr_ring_root", "dr_ring_prove_batch", "dr_ring_verify_batch", "dr_ring_verify_set_msm_threshold", "dr_last_error"):
        getattr(lib.lib, name)
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


def coeffs(n, agg):
    r = random.Random(n)
    return [v for _ in range(n) for v in ((r.randrange(1, fr.R) if agg else 1), r.randrange(1, fr.R))]


MODES = [("per_item", False, 8192), ("aggregate", True, 8192), ("aggregate_msm", True, 1)]


def prove(ring, r, cnt):
    rng = random.Random(r)
    al = [b"probe-input-%d-" % r + le64(j) for j in range(cnt)]
    ad = [b"probe-ad-%d-" % r + le64(j) for j in range(cnt)]
    pr, st = ring.prove_batch(al, ad, [sk] * cnt, [3] * cnt, zk_rows=[rng.randrange(fr.R) for _ in range(12 * cnt)])
    assert not any(st)
    return pr, al, ad


if AB_ONLY:  # ---- no regression, one library: dr_ring_verify_batch of 4096 proofs in every mode
    srs = native_srs(ctx, None, WINDOW_BITS)
    ring = native_ring(srs, ring_keys(0), params)
    pr, al, ad = prove(ring, 0, N)
    res = {}
    for name, agg, thr in MODES:
        co = coeffs(N, agg)
        lib.lib.dr_ring_verify_set_msm_threshold(thr)
        dev_ms, wall_ms = [], []
        for rep in range(REPS + 1):
            (v, ok), dev, wall = timed(ctx, lambda: ring.verify_batch(al, ad, pr, co, aggregate=agg))
            assert ok and v == [1] * N, name
            if rep:  # rep 0 warms up
                dev_ms.append(dev)
                wall_ms.append(wall)
        lib.lib.dr_ring_verify_set_msm_threshold(8192)
        res[name] = {"device_ms": dev_ms, "wall_ms": wall_ms}
    print("AB_RESULT " + json.dumps(res), flush=True)
    sys.exit(0)

# ---- verifier cost ------------------------------------------------------------------------------------------------------
free0 = ctx.device_info()["free_bytes"]
t0 = time.perf_counter()
srs = native_srs(ctx, None, WINDOW_BITS)
ctx.sync()
t_srs = time.perf_counter() - t0
t0 = time.perf_counter()
rings = [native_ring(srs, ring_keys(0), params)]
ctx.sync()
t_ring = time.perf_counter() - t0
free1 = ctx.device_info()["free_bytes"]
root0 = rings[0].root()
verifier_ms = []
for _ in range(REPS):
    t0 = time.perf_counter()
    v = make_verifier(ctx, root0, params)
    verifier_ms.append((time.perf_counter() - t0) * 1e3)
    v.close()
free2 = ctx.device_info()["free_bytes"]
vs = [make_verifier(ctx, root0, params) for _ in range(64)]
free3 = ctx.device_info()["free_bytes"]
for v in vs:
    v.close()
out["verifier_cost"] = {
    "srs_load_s (window table, %d bits)" % WINDOW_BITS: t_srs, "ring_create_s": t_ring, "srs_plus_ring_device_bytes": free0 - free1,
    "verifier_create_ms": stats(verifier_ms), "device_bytes_64_verifiers (free-memory delta)": free2 - free3,
}
print(out["verifier_cost"], flush=True)

# ---- no regression: dr_ring_verify_batch, this tree's library and the parent's, alternated processes -------------------------
runs = {"branch": str(_native.DEFAULT_LIBRARY)}
if len(sys.argv) > 1:
    runs["parent"] = sys.argv[1]
ab = {k: {name: {"device_ms": [], "wall_ms": []} for name, _, _ in MODES} for k in runs}
for rep in range(int(os.environ.get("AB_PROCESSES", "3"))):
    for k in (list(runs) if rep % 2 == 0 else list(runs)[::-1]):
        proc = subprocess.run([sys.executable, os.path.abspath(__file__), "--ab", runs[k]], capture_output=True, text=True, timeout=300)
        line = [x for x in proc.stdout.splitlines() if x.startswith("AB_RESULT ")]
        assert proc.returncode == 0 and line, (k, proc.stdout[-2000:], proc.stderr[-2000:])
        for name, d in json.loads(line[0][len("AB_RESULT "):]).items():
            for m, xs in d.items():
                ab[k][name][m] += xs
        print(k, rep, flush=True)
out["verify_batch_4096_ring1023"] = {k: {name: {m: stats(xs) for m, xs in d.items()} for name, d in per.items()} for k, per in ab.items()}
for name, _, _ in MODES:
    print(name, {k: out["verify_batch_4096_ring1023"][k][name]["device_ms"]["median"] for k in runs}, flush=True)

# ---- proofs for the multi-ring runs: ring 0 4096, rings 1..7 512 each, rings 8..63 64 each --------------------------------------
rings += [native_ring(srs, ring_keys(r), params) for r in range(1, 64)]
proofs, alphas, ads = {}, {}, {}
for r, cnt in [(0, N)] + [(r, 512) for r in range(1, 8)] + [(r, 64) for r in range(8, 64)]:
    proofs[r], alphas[r], ads[r] = prove(rings[r], r, cnt)
print("proved", flush=True)

# ---- gain: one multi call vs K dr_ring_verify_batch calls ------------------------------------------------------------------
gain = {}
for K in (1, 8, 64):
    per = N // K
    members = list(range(K))
    al = [a for r in members for a in alphas[r][:per]]
    ad = [d for r in members for d in ads[r][:per]]
    pr = [p for r in members for p in proofs[r][:per]]
    index = [r for r in members for _ in range(per)]
    verifiers = [make_verifier(ctx, rings[r].root(), params) for r in members]
    for name, agg, thr in MODES:
        co = coeffs(N, agg)
        ctx.library.lib.dr_ring_verify_set_msm_threshold(thr)
        multi_dev, multi_wall, loop_dev, loop_wall = [], [], [], []
        for rep in range(REPS + 1):
            (v, ok), dev, wall = timed(ctx, lambda: _native.NativeRingVerifier.verify_multi(verifiers, index, al, ad, pr, co, agg))
            assert ok and v == [1] * N, (K, name)
            if rep:
                multi_dev.append(dev)
                multi_wall.append(wall)

            def loop():
                res = [rings[r].verify_batch(al[r * per : (r + 1) * per], ad[r * per : (r + 1) * per], pr[r * per : (r + 1) * per], co[2 * r * per : 2 * (r + 1) * per], agg)
                       for r in members]
                return res

            res, dev, wall = timed(ctx, loop)
            assert all(ok and v == [1] * per for v, ok in res), (K, name)
            if rep:
                loop_dev.append(dev)
                loop_wall.append(wall)
        ctx.library.lib.dr_ring_verify_set_msm_threshold(8192)
        gain[f"K{K}_{name}"] = {"multi_device_ms": stats(multi_dev), "multi_wall_ms": stats(multi_wall), "loop_device_ms": stats(loop_dev), "loop_wall_ms": stats(loop_wall)}
        print(K, name, gain[f"K{K}_{name}"]["multi_device_ms"]["median"], gain[f"K{K}_{name}"]["loop_device_ms"]["median"], flush=True)
    for v in verifiers:
        v.close()
out["multi_vs_loop_4096"] = gain
path = os.environ.get("PROBE_OUT") or os.path.join(tempfile.gettempdir(), "probe_ring_verifier.json")
os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
with open(path, "w") as f:
    json.dump(out, f, indent=1)
print("wrote", path, flush=True)
print(json.dumps({k: v for k, v in out.items() if k == "nvidia_smi"}))
