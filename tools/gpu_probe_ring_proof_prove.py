#!/usr/bin/env python
"""GPU probe: bare ring proofs from a caller's blinding factor (dr_ring_proof_prove_multi); writes its results as JSON to $PROBE_OUT
(default: probe_ring_proof_prove.json in the temporary directory).

  python tools/gpu_probe_ring_proof_prove.py [PARENT_LIB]
  python tools/gpu_probe_ring_proof_prove.py --ptxas     (registers and spills of RingProofStartBody; needs nvcc, no GPU)

- no regression: dr_ring_prove_batch of 4096 proofs at ring 1023 with the bench's default table (16-bit windows over GLV halves), with
  this tree's library and (when PARENT_LIB, a build of the parent commit, is given) that library: one process per library and run,
  the processes alternated, each timing REPS calls after a warm-up call; the first and last proof must agree;
- the bare prover: 4096 proofs at ring 1023 on the same rows, blinding factors and zk rows as the dr_ring_prove_batch call it is
  timed next to (alternated within one process), its payloads checked against bytes 192..784 of those proofs; and 4096 bare proofs
  over K = 8 rings of 1023 keys in one call;
- the per-phase split (dr_ring_prove_phase_ms) of both provers.
Times are device times (CUDA events on the context stream around the whole call).  The card's name, power limit and maximum SM clock
are read in the same run."""
import ctypes
import json
import os
import random
import re
import subprocess
import sys
import tempfile
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

if len(sys.argv) > 1 and sys.argv[1] == "--ptxas":  # compile-only: the start kernel's registers, spills and stack
    with tempfile.TemporaryDirectory() as tmp:
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        proc = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--extended-lambda", "-Xcompiler", "-fPIC", "-Xptxas", "-v",
                               "-c", os.path.join(ROOT, "dot_ring_b200", "csrc", "api_ring.cu"), "-o", os.path.join(tmp, "api_ring.o")],
                              capture_output=True, text=True, check=True)  # fmt: skip
    lines = proc.stderr.splitlines()
    report = {}
    for name in ("RingProofStartBody", "PedersenStartBody"):
        for i, line in enumerate(lines):
            if "Compiling entry function" in line and name in line:
                block = " ".join(lines[i + 1 : i + 4])
                regs = re.search(r"Used (\d+) registers", block)
                spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", block)
                stack = re.search(r"(\d+) bytes stack frame", block)
                report[name] = {"registers": int(regs.group(1)) if regs else None, "spill_stores": int(spill.group(1)) if spill else None,
                                "spill_loads": int(spill.group(2)) if spill else None, "stack_frame": int(stack.group(1)) if stack else None}
                break
    print(json.dumps(report))
    sys.exit(0)

from dot_ring_b200 import _native  # noqa: E402
from dot_ring_b200.srs import read_srs_file  # noqa: E402
from oracle import bandersnatch as bs  # noqa: E402
from oracle import fr, ring_proof as rp  # noqa: E402
from oracle import transcript as otr  # noqa: E402
from tests.helpers import bench_ring_keys, le64, seed  # noqa: E402
from tests.ring_fixtures import native_ring  # noqa: E402
from tests.verify_cases import suite_struct  # noqa: E402

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
    """ctypes library view for _declare on a parent build: entry points it lacks (dr_ring_proof_prove_multi) are skipped."""

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
    c.timer_start()
    res = fn()
    return res, c.timer_stop()


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
    dev_ms, first = [], None
    for rep in range(REPS + 1):
        (pr, st), dev = timed(ctx, lambda: ring.prove_batch(al, ad, [sk] * N, [3] * N, zk_rows=zk))
        assert not any(st)
        first = first or pr[0] + pr[-1]
        if rep:  # rep 0 warms up
            dev_ms.append(dev)
    print("AB_RESULT " + json.dumps({"device_ms": dev_ms, "first_last_proof": first.hex()}), flush=True)
    sys.exit(0)

# ---- no regression: dr_ring_prove_batch, this tree's library and the parent's, alternated processes ------------------------------
runs = {"branch": str(_native.DEFAULT_LIBRARY)}
if len(sys.argv) > 1:
    runs["parent"] = sys.argv[1]
ab = {k: {"device_ms": [], "first_last_proof": set()} for k in runs}
for rep in range(int(os.environ.get("AB_PROCESSES", "4"))):
    for k in (list(runs) if rep % 2 == 0 else list(runs)[::-1]):
        proc = subprocess.run([sys.executable, os.path.abspath(__file__), "--ab", runs[k]], capture_output=True, text=True, timeout=600)
        line = [x for x in proc.stdout.splitlines() if x.startswith("AB_RESULT ")]
        assert proc.returncode == 0 and line, (k, proc.stdout[-2000:], proc.stderr[-2000:])
        d = json.loads(line[0][len("AB_RESULT "):])
        ab[k]["device_ms"] += d["device_ms"]
        ab[k]["first_last_proof"].add(d["first_last_proof"])
        print(k, rep, stats(d["device_ms"])["median"], flush=True)
out["prove_batch_4096_ring1023"] = {k: {"device_ms": stats(v["device_ms"])} for k, v in ab.items()}
out["same_proofs_as_parent"] = len(set().union(*[v["first_last_proof"] for v in ab.values()])) == 1
print({k: out["prove_batch_4096_ring1023"][k]["device_ms"]["median"] for k in runs}, "same proofs:", out["same_proofs_as_parent"], flush=True)

# ---- bare prover next to dr_ring_prove_batch on the same rows --------------------------------------------------------------------
srs = bench_srs(ctx)
rings = [native_ring(srs, ring_keys(r), params) for r in range(8)]
al, ad, zk = batch(0, N)
ts = ctx.pedersen_prove_with_blinding(suite_struct(), al, ad, [sk] * N)[1]
fused_ms, bare_ms, fused_phase, bare_phase = [], [], [], []
for rep in range(REPS + 1):
    (pr, st), dev = timed(ctx, lambda: rings[0].prove_batch(al, ad, [sk] * N, [3] * N, zk_rows=zk))
    assert not any(st)
    phase_f = rings[0].prove_phase_ms()
    (rel, pay), dev_b = timed(ctx, lambda: _native.NativeRing.proof_prove_multi([rings[0]], [0] * N, [3] * N, ts, zk))
    phase_b = rings[0].prove_phase_ms()
    if rep == 0:
        assert pay == [p[192:] for p in pr], "bare payloads differ from the Ring VRF proofs"
        assert rel == [bs.dec_point(p[32:64]) for p in pr], "relations differ from the blinded keys"
        continue
    fused_ms.append(dev)
    bare_ms.append(dev_b)
    fused_phase.append(phase_f)
    bare_phase.append(phase_b)
out["one_ring_4096"] = {"prove_batch_device_ms": stats(fused_ms), "bare_device_ms": stats(bare_ms), "prove_batch_phase_ms": fused_phase[len(fused_phase) // 2],
                        "bare_phase_ms": bare_phase[len(bare_phase) // 2],
                        "phase_order": "pedersen+witness, interpolate, commits, LDE+constraints+quotient, evaluations+openings, transcripts+assembly"}
print("one ring 4096: prove_batch", stats(fused_ms)["median"], "bare", stats(bare_ms)["median"], flush=True)

# ---- bare prover over K = 8 rings ------------------------------------------------------------------------------------------------
index = [j % 8 for j in range(N)]
k8 = []
for rep in range(REPS + 1):
    _, dev = timed(ctx, lambda: _native.NativeRing.proof_prove_multi(rings, index, [3] * N, ts, zk))
    if rep:
        k8.append(dev)
out["eight_rings_4096_bare_device_ms"] = stats(k8)
print("eight rings 4096 bare", stats(k8)["median"], flush=True)

path = os.environ.get("PROBE_OUT") or os.path.join(tempfile.gettempdir(), "probe_ring_proof_prove.json")
os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
with open(path, "w") as f:
    json.dump(out, f, indent=1)
print("wrote", path, flush=True)
