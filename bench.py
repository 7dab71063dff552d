#!/usr/bin/env python
"""Headline benchmark: Ring VRF proofs/s at ring size 1023 (domain 2^11), batched on B200.

    python bench.py --gpus N --steps K --warmup W            # this engine
    python bench.py --impl reference --gpus N --steps K ...   # reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's proofs as DIR/*.npy

Workload (BASELINE.json configs[1]; seeding of the reference's own tests/benchmark/bench_ring_proof.py:
47-77,140-152): one 1023-key ring, signer at index 3, per step ONE batch of `--total` (4096) proofs with
alpha = "bench-batch-input" | le64(j), ad = "bench-batch-ad" | le64(j) and 12 blinding rows per proof from
random.Random(step), sharded contiguously over the GPUs (strong scaling, no data-path collective): under torchrun
every rank proves its slice of the batch; `python bench.py --gpus N` without torchrun drives N GPUs from one process
through dot_ring_b200.engine.EnginePool.  `--batch B` selects weak scaling instead (B proofs per GPU per step); the
strong line also carries that operating point as `saturated` (8192 proofs per GPU per step).
`value` = proofs of all GPUs / max-over-ranks device time (one CUDA event pair around each step's call);
`e2e` = the same through the public Python API with host buffers (H2D of the inputs and D2H of the 784-byte
proofs inside the timed region).

Before anything is timed the six ring-1023 proofs of the unmodified reference (tests/golden/ring1023_reference.json)
are proved through the same engine, window table and batch width and compared byte for byte; after the timed region a
sample of the last step's proofs is verified on the device (and, at N=1, three of them by the CPU oracle inside the
cpu_baseline leg).  No value is printed if any of that fails.

A number printed by this script under a profiler is not a bench value.
"""

from __future__ import annotations

import argparse
import gc
import hashlib
import json
import os
import random
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

FR = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
RING_SIZE = 1023
SIGNER_INDEX = 3
MSM_SIZES = (2048, 2048, 2048, 2048, 6145, 6144, 2047)  # per proof at N = 2048 (SURVEY.md 3.2)
DENSE_MSM_SIZES = (6145, 6144, 2047)  # quotient + two openings: dense coefficient vectors
def sparse_witness_madds(table_bits: int) -> int:
    """Witness columns are committed from their evaluation form: ~131.5 non-zero steps for acc_x / acc_y (one table addition per
    window each), ~135 unit steps for b, 1 for acc_ip, plus 3 blinding rows per column."""
    w = -(-256 // max(table_bits, 1))
    return int(2 * 131.5 * w + 135 + 3 * w + 1 + 4 * w)


def seed_bytes(*parts) -> bytes:
    h = hashlib.sha256()
    for part in parts:
        if isinstance(part, bytes):
            h.update(part)
        elif isinstance(part, int):
            h.update(part.to_bytes(8, "little"))
        else:
            h.update(part.encode())
        h.update(b"\0")
    return h.digest()


def le64(i: int) -> bytes:
    return i.to_bytes(8, "little")


def canonical_fq_mul_per_msm(n: int) -> int:
    """SURVEY.md 8(d): Pippenger, signed c-bit windows: min_c ceil(255/c) * (n*10 + 2^c*14) Fq multiplications."""
    return min(-(-255 // c) * (n * 10 + (1 << c) * 14) for c in range(2, 21))


CANONICAL_IMAD_PER_PROOF = sum(canonical_fq_mul_per_msm(n) for n in MSM_SIZES) * 600  # 600 IMAD per 12-limb Montgomery mul
# executed by one XYZZ mixed addition: 8 multiplications (600 IMAD each, the CIOS word-product count) + 2 squarings (456: the cross
# products are formed once, tools/gen_field_asm.py prog_sqr)
MADD_IMAD = 8 * 600 + 2 * 456


class ClockSampler(threading.Thread):
    """SM clock, power and throttle reasons sampled during the timed region: NVML in-process (no child process next to the
    timed calls); `nvidia-smi` only when the NVML binding is missing."""

    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, device: int):
        super().__init__(daemon=True)
        visible = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        ids = [v.strip() for v in visible.split(",") if v.strip()]
        self.device = int(ids[device]) if device < len(ids) and ids[device].isdigit() else device
        self.samples: list[dict] = []
        self._halt = threading.Event()

    def _nvml_loop(self) -> bool:
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.device)
            sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            return False
        while not self._halt.is_set():
            try:
                mask = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.samples.append({
                    "sm": float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), "max": sm_max, "power": pynvml.nvmlDeviceGetPowerUsage(h) / 1e3,
                    "reasons": ["Active" if mask & bit else "Not Active" for bit, _ in self.REASONS],
                })  # fmt: skip
            except Exception:
                pass
            self._halt.wait(0.1)
        return True

    def run(self) -> None:
        if self._nvml_loop():
            return
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self._halt.is_set():
            try:
                out = subprocess.run(
                    ["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}", "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5
                ).stdout.strip()
                f = [x.strip() for x in out.split(",")]
                if len(f) >= 7:
                    self.samples.append({"sm": float(f[0]), "max": float(f[1]), "power": float(f[2]), "reasons": f[3:7]})
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self) -> dict:
        self._halt.set()
        self.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(s["sm"] for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i, r in enumerate(s["reasons"]) if r.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.samples[0]["max"], "power_w_max": max(s["power"] for s in self.samples), "reasons": reasons, "samples": len(sm)}


DRY_RUN = os.environ.get("DOT_RING_B200_BENCH_DRYRUN") == "1"  # tests only: CPU emulation build + gloo


def dist_setup(n_gpus: int):
    """One process per GPU; torch.distributed (NCCL) is plumbing for the barrier and the max-over-ranks only."""
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world <= 1:
        return rank, local, 1, None
    import torch
    import torch.distributed as dist

    if DRY_RUN:
        dist.init_process_group(backend="gloo")
        return rank, local, world, dist
    torch.cuda.set_device(local)
    dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    return rank, local, world, dist


def _device(local):
    import torch

    return torch.device("cpu") if DRY_RUN else torch.device("cuda", local)


def barrier(dist, local):
    if dist is not None:
        import torch

        if DRY_RUN:
            dist.barrier()
            return
        dist.barrier(device_ids=[local])
        torch.cuda.synchronize()


def _reduce(dist, local, values: list[float], op) -> list[float]:
    if dist is None:
        return values
    import torch

    t = torch.tensor(values, dtype=torch.float64, device=_device(local))
    dist.all_reduce(t, op=op)
    return [float(x) for x in t.tolist()]


def reduce_max(dist, local, values: list[float]) -> list[float]:
    return _reduce(dist, local, values, None if dist is None else dist.ReduceOp.MAX)


def reduce_sum(dist, local, values: list[float]) -> list[float]:
    return _reduce(dist, local, values, None if dist is None else dist.ReduceOp.SUM)


# -------------------------------------------------------------------------------------------------- ours
GOLDEN_RING1023 = ROOT / "tests" / "golden" / "ring1023_reference.json"  # written by the unmodified reference (tests/golden/generate_golden.py)


def build_engine(args, local: int, n_local_devices: int, dry_run: bool):
    """Engine (one device) or EnginePool (one process, several devices) with the requested window table; falls back to the next
    smaller geometry when the device cannot hold it.  Returns (engine, seconds)."""
    from dot_ring_b200 import engine as eng_mod

    t0 = time.perf_counter()
    library = None
    if dry_run:
        from tests.host.emul import emulation_library

        library = emulation_library()
    requested = (args.window_bits, args.wide_windows, bool(args.glv))
    size = lambda g: (-(-((128 if g[2] else 256) - g[1]) // g[0]) + g[1]) << (g[0] - 1) if g[0] else 0  # ~table entries per SRS point  # noqa: E731
    candidates = [requested] + [g for g in ((14, 4, False), (14, 0, False), (13, 0, False), (12, 0, False)) if size(g) < size(requested)]

    def one(device: int):
        eng = eng_mod.Engine(device, window_bits=args.window_bits, library=library, wide_windows=args.wide_windows, glv=bool(args.glv))
        if not dry_run and not eng.ctx.library.is_cuda:
            raise SystemExit("bench.py measures the CUDA build only")
        for idx, (c, k, glv) in enumerate(candidates):
            eng.window_bits, eng.wide_windows, eng.glv = c, k, glv
            try:
                _ = eng.srs
                # the ring tables (2.6 GB) and a 4096-proof pass (9.5 GB) must still fit next to the table
                left = eng.ctx.device_info()["free_bytes"]
                if not dry_run and left < 14e9 and idx + 1 < len(candidates):
                    print(f"[bench] window table ({c}, {k}, glv={glv}) leaves only {left / 1e9:.1f} GB: falling back", file=sys.stderr, flush=True)
                    eng._srs.close()
                    eng._srs = None
                    eng.ctx.trim()
                    continue
                break
            except MemoryError as e:
                print(f"[bench] window table ({c}, {k}, glv={glv}) does not fit: {e}", file=sys.stderr, flush=True)
                eng.ctx.trim()
        else:
            raise SystemExit("bench.py: no window table fits on this device")
        eng.ctx.set_commit_mode(args.commit_mode)
        if args.prove_chunk:
            eng.ctx.set_prove_chunk(args.prove_chunk)
        eng.ctx.sync()
        return eng

    if n_local_devices <= 1:
        eng = one(local)
        eng_mod.set_default_engine(eng, local)
        return eng, time.perf_counter() - t0
    pool = eng_mod.EnginePool.__new__(eng_mod.EnginePool)  # engines built by `one` (table fallback per device), then adopted by the pool
    from concurrent.futures import ThreadPoolExecutor

    pool.devices = [0] * n_local_devices if dry_run else list(range(n_local_devices))
    pool._workers = [ThreadPoolExecutor(max_workers=1, thread_name_prefix=f"dr-gpu{d}") for d in pool.devices]
    pool.engines = pool.map(lambda i: one(pool.devices[i]))
    pool.ctx = eng_mod.PooledContext(pool)
    pool.srs_bytes = pool.engines[0].srs_bytes
    eng_mod.set_default_engine(pool, local)
    return pool, time.perf_counter() - t0


def golden_parity(RingVRF, Bandersnatch, ring, sk, pk, width: int, keys: list[bytes], rng, limit: int | None = None) -> dict:
    """Prove, in ONE batch of the bench's own per-device width through the bench's engine / table / ring, the six ring-1023 proofs
    the unmodified reference produced (4 with zeroed blinding rows, 2 with given rows) and compare the 784 bytes of each."""
    g = json.loads(GOLDEN_RING1023.read_text())
    if hashlib.sha256(b"".join(keys)).hexdigest() != g["keys_sha256"] or pk.hex() != g["signer_pk"]:
        raise SystemExit("bench.py: the synthetic ring differs from the reference's benchmark ring (tests/golden/ring1023_reference.json)")
    items = [(bytes.fromhex(v["alpha"]), bytes.fromhex(v["ad"]), [0] * 12, v["proof"]) for v in g["proofs_test_vectors"][:limit]]
    items += [(bytes.fromhex(v["alpha"]), bytes.fromhex(v["ad"]), [int(z, 16) for z in v["zk_rows"]], v["proof"]) for v in g["proofs_blinded"][:limit]]
    n = max(width, len(items))
    alphas = [it[0] for it in items] + [b"bench-parity-filler" + le64(j) for j in range(n - len(items))]
    ads = [it[1] for it in items] + [b"" for _ in range(n - len(items))]
    zk = b"".join(z.to_bytes(32, "little") for it in items for z in it[2]) + b"".join(rng.randrange(FR).to_bytes(32, "little") for _ in range(12 * (n - len(items))))
    proofs = RingVRF[Bandersnatch].prove_batch(alphas, ads, sk, pk, ring, None, zk_rows=zk, as_bytes=True)
    equal = [proofs[i].hex() == it[3] for i, it in enumerate(items)]
    if not all(equal):
        raise SystemExit(f"bench.py: golden proofs differ from the reference at items {[i for i, e in enumerate(equal) if not e]}; refusing to report a number")
    return {"golden_proofs": len(items), "equal": True, "batch_width": n}


def run_ours(args) -> None:
    rank, local, world, dist = dist_setup(args.gpus)
    pool_devices = args.gpus if world == 1 and args.gpus > 1 else 1  # one process driving several GPUs through EnginePool
    n_dev = world * pool_devices
    os.environ["DOT_RING_B200_DEVICE"] = str(local)
    from dot_ring_b200 import Bandersnatch, Ring, RingProofParams, RingRoot, RingVRF

    dry_run = DRY_RUN
    eng, table_s = build_engine(args, local, pool_devices, dry_run)
    engines = eng.engines if pool_devices > 1 else [eng]
    info = engines[0].ctx.device_info()
    lib = engines[0].ctx.library

    # synthetic ring: keys derived with the product's own key derivation (no oracle on this path)
    t0 = time.perf_counter()
    seeds = [seed_bytes("batch-signer", 0, 0) if i == SIGNER_INDEX else seed_bytes("ring-member", 0, i) for i in range(RING_SIZE)]
    from dot_ring_b200.transcript import secret_scalar_from_seed

    sks = [secret_scalar_from_seed(Bandersnatch, s).to_bytes(32, "little") for s in seeds]
    keys = Bandersnatch.public_keys_from_secrets(sks)
    sk, pk = sks[SIGNER_INDEX], keys[SIGNER_INDEX]
    params = RingProofParams.from_ring_size(RING_SIZE)
    ring = Ring(keys, params, eng)
    root = RingRoot.from_ring(ring, params)
    root_bytes = root.encode()
    ring_s = time.perf_counter() - t0
    ring.native.time_calls = True
    prove = lambda a, d, zk: RingVRF[Bandersnatch].prove_batch(a, d, sk, pk, ring, None, zk_rows=zk, as_bytes=True)  # noqa: E731

    # ---- workload ---------------------------------------------------------------------------------------------
    strong = args.scaling == "strong"
    if strong:  # BASELINE configs[1]: ONE batch of `total` proofs per step, sharded contiguously over the GPUs
        total = args.total
        lo, hi = _shard(total, world, rank)
    else:  # every GPU proves its own `batch` proofs per step
        total = args.batch * n_dev
        lo, hi = rank * args.batch * pool_devices, (rank + 1) * args.batch * pool_devices
    mine = hi - lo
    per_device = -(-mine // pool_devices)

    def inputs(step: int, lo: int, hi: int, total: int, stream_seed):
        """alpha / ad = the reference's benchmark strings over the global proof index j = step * total + g; blinding rows from
        random.Random(stream_seed): in strong mode ONE stream over the whole batch (SURVEY 8d config 2), sliced per rank."""
        rng = random.Random(stream_seed)
        if lo:
            for _ in range(12 * lo):
                rng.randrange(FR)
        base = step * total
        return (
            [b"bench-batch-input" + le64(base + g) for g in range(lo, hi)],
            [b"bench-batch-ad" + le64(base + g) for g in range(lo, hi)],
            b"".join(rng.randrange(FR).to_bytes(32, "little") for _ in range(12 * (hi - lo))),  # blinding rows as wire bytes
        )

    # ---- parity gate: the reference's own proofs through this engine, table and batch width -------------------
    parity = golden_parity(RingVRF, Bandersnatch, ring, sk, pk, mine, keys, random.Random(1234 + rank), limit=1 if dry_run else None)
    parity["ring_root_sha256"] = hashlib.sha256(root_bytes).hexdigest()[:16]

    # the prepared inputs are a few hundred thousand small Python objects: keep the cyclic collector from rescanning them in the
    # middle of a timed step (a generation-2 pass costs 10 - 30 ms)
    gc.collect()
    gc.freeze()
    launches0 = lib.launch_count()
    for w in range(args.warmup):
        a, d, zk = inputs(500_000 + w, lo, hi, total, (w + 1) * 7919 if strong else 1_000_003 * (rank + 1) + w)
        prove(a, d, zk)
    launches_warm = lib.launch_count()

    prepared = [inputs(s, lo, hi, total, s if strong else 1_000_003 * (rank + 1) + 1000 + s) for s in range(args.steps)]
    gc.collect()
    gc.freeze()
    sampler = ClockSampler(local)
    sampler.start()
    barrier(dist, local)
    for e in engines:
        e.ctx.sync()
    dev_ms, phases, kernel_ms, kernel_launches = 0.0, [0.0] * 6, 0.0, 0
    step_ms = []
    t_start = time.perf_counter()
    last = None
    for a, d, zk in prepared:
        last = prove(a, d, zk)
        dev_ms += ring.native.last_call_ms  # one CUDA event pair around the whole call (slowest device of a pool)
        step_ms.append(round(ring.native.last_call_ms, 3))
        ph = ring.native.prove_phase_ms()
        phases = [x + y for x, y in zip(phases, ph)]
        km, kl = ring.native.commit_kernel_ms()
        kernel_ms += km
        kernel_launches += kl
    for e in engines:
        e.ctx.sync()
    barrier(dist, local)
    wall_s = time.perf_counter() - t_start
    clocks = sampler.stop()
    launches = lib.launch_count() - launches_warm

    # ---- every timed step's output is checked: a sample of the last step with the device verifier -------------
    la, ld, _ = prepared[-1]
    k = min(len(last), 64)
    picks = sorted(random.Random(99).sample(range(len(last)), k))
    verdicts = RingVRF[Bandersnatch].verify_batch([last[i] for i in picks], [la[i] for i in picks], [ld[i] for i in picks], ring, root)
    if verdicts != [1] * k or len(set(last)) != len(last):
        raise SystemExit("bench.py: proofs of the timed region do not verify; refusing to report a number")
    parity["verified_sample"] = k
    oracle_sample = [(last[i], la[i], ld[i]) for i in picks[:3]]
    if args.dump_outputs:
        dump_outputs(Path(args.dump_outputs), last, lo, "proofs" if world == 1 else f"proofs_rank{rank}", world)

    # integer-pipe ceiling measured live on this GPU (dependent-free mad.lo.u32, all SMs)
    if dry_run:
        imad_peak = imad_wide_peak = 148 * 64 * 1.965e9  # nominal; a dry run is not a measurement
    else:
        imad_peak, _ = engines[0].ctx.microbench("imad", 20000)
        imad_wide_peak, _ = engines[0].ctx.microbench("imad_wide", 20000)

    # ---- the other operating point, reported beside the headline: every GPU saturated with its own 8192-proof passes ----
    saturated = None
    if strong and args.saturated_batch and not dry_run:
        sb = args.saturated_batch * pool_devices
        slo = rank * sb
        for w in range(2):
            prove(*inputs(700_000 + w, slo, slo + sb, sb * world, 1_000_003 * (rank + 1) + 2000 + w))
        sat_in = [inputs(710_000 + s, slo, slo + sb, sb * world, 1_000_003 * (rank + 1) + 3000 + s) for s in range(args.saturated_steps)]
        barrier(dist, local)
        sat_ms, t1 = 0.0, time.perf_counter()
        for a, d, zk in sat_in:
            prove(a, d, zk)
            sat_ms += ring.native.last_call_ms
        barrier(dist, local)
        sat_wall = time.perf_counter() - t1
        smx = reduce_max(dist, local, [sat_ms, sat_wall])
        n_sat = sb * world * args.saturated_steps
        saturated = {"proofs_per_gpu_per_step": args.saturated_batch, "steps": args.saturated_steps, "value": n_sat / (smx[0] * 1e-3), "e2e": n_sat / smx[1], "unit": "proofs/s",
                     "scaling": "weak", "note": "every GPU proves its own full-width passes (the throughput operating point of round 1's headline)"}

    mx = reduce_max(dist, local, [dev_ms, wall_s])
    proofs_total = total * args.steps
    value = proofs_total / (mx[0] * 1e-3)
    e2e = proofs_total / mx[1]
    window_bits, wide_windows, glv, windows = engines[0].srs.geometry
    wbits = ring.native.witness_table_bits() or 10
    # dominant kernel = the dense fixed-base commit (quotient + two openings); event-timed around its launches only
    dense_madds = sum(DENSE_MSM_SIZES) * windows
    kernel_imad = dense_madds * MADD_IMAD * mine * args.steps / pool_devices  # per device
    kernel_rate = kernel_imad / (kernel_ms * 1e-3) if kernel_ms else 0.0
    canonical_dense = sum(canonical_fq_mul_per_msm(n) for n in DENSE_MSM_SIZES) * 600
    madds_per_proof = dense_madds + sparse_witness_madds(wbits)
    step_imad = madds_per_proof * MADD_IMAD * mine * args.steps / pool_devices
    table_bytes_per_launch = dense_madds * 96 * per_device / 3  # average over the 3 launches of a pass

    if dist is not None:
        dist.destroy_process_group()
    if rank != 0:
        return
    per_gpu = total // n_dev if strong else args.batch
    line = {
        "metric": "ring_vrf_proofs_per_s",
        "value": value,
        "unit": "proofs/s",
        "n_gpus": n_dev,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": mx[0] / args.steps,
        "higher_is_better": True,
        "scaling": "strong" if strong else "weak",
        "vs_baseline": None,
        "dtype": "u32 limbs (381-bit Fq / 255-bit Fr Montgomery)",
        "data": "synthetic",
        "config": {
            "workload": workload_string(strong, total, n_dev, args.batch),
            "total_proofs_per_step": total,
            "proofs_per_gpu_per_step": per_gpu,
            "launch": "one process, EnginePool over %d devices" % pool_devices if pool_devices > 1 else ("torchrun, one rank per GPU" if world > 1 else "one process, one GPU"),
            "window_bits": window_bits,
            "wide_windows": wide_windows,
            "glv_split": bool(glv),
            "table_additions_per_coefficient": windows,
            "table_gb": round(engines[0].srs.table_bytes / 1e9, 2),
            "l2": "per-step working set (window table + ~2 MB of scratch per proof) is far larger than the 126 MB L2; no flush needed",
            "parity": parity,
        },
        "e2e": {"value": e2e, "unit": "proofs/s", "h2d_bytes_per_step": total * (12 * 32 + 32 + 4 * 5 + 25 + 22), "d2h_bytes_per_step": total * (784 + 4), "ms_per_step": mx[1] * 1e3 / args.steps},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {
            "kernel": "kernel_entry_lb<CommitBodyT<GLV>> (dense fixed-base KZG commit: quotient + two openings)",
            "bound": "imad (int32 multiply-add pipe; neither hbm nor tensor: the path is 381-bit modular arithmetic)",
            "achieved": kernel_rate / 1e12,
            "peak": imad_peak / 1e12,
            "unit": "T IMAD/s executed by the kernel (mixed G1 additions issued x (8 mul x 600 + 2 sqr x 456) IMAD), CUDA events around its launches only",
            "frac": kernel_rate / imad_peak,
            "kernel_ms_per_step": kernel_ms / args.steps,
            "kernel_launches_per_step": kernel_launches / args.steps,
            "kernel_share_of_step": kernel_ms / dev_ms if dev_ms else None,
            "algorithmic_reduction": canonical_dense / (dense_madds * MADD_IMAD),
            "algorithmic_reduction_note": "canonical Pippenger IMAD of the same three MSMs (SURVEY.md 8d) / IMAD executed: the fixed-base table removes buckets and doublings",
            "whole_step_executed_frac": step_imad / (dev_ms * 1e-3) / imad_peak if dev_ms else None,
            "whole_step_canonical_frac": CANONICAL_IMAD_PER_PROOF * mine * args.steps / pool_devices / (dev_ms * 1e-3) / imad_peak if dev_ms else None,
            "peak_source": "measured live: dependent-free mad.lo.u32 on all SMs (dr_microbench); IMAD.WIDE measured " + f"{imad_wide_peak / 1e12:.2f} T/s",
            "traffic": NCU_TRAFFIC["glv" if glv else "plain"]["bytes"],
            "traffic_launch": NCU_TRAFFIC["glv" if glv else "plain"]["launch"],
            "algorithmic_table_bytes_per_launch": table_bytes_per_launch,
            "hbm_gbs_for_table_reads": dense_madds * 96 * mine * args.steps / pool_devices / (kernel_ms * 1e-3) / 1e9 if kernel_ms else None,
        },
        "step_ms_rank0": step_ms,
        "phase_ms_per_step": {k: v / args.steps for k, v in zip(["pedersen+witness", "interpolate", "commit(msm)", "lde+constraints+quotient", "evals+openings", "transcripts+assembly"], phases)},
        "setup": {"srs_table_s": table_s, "ring_s": ring_s, "device": info["name"], "sm_count": info["sm_count"]},
    }
    if saturated:
        line["saturated"] = saturated
    if dry_run:
        line["dry_run"] = "CPU emulation of the kernels (tests only); not a measurement"
    if n_dev == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_single(oracle_sample)
        line["config"]["parity"]["oracle_verified"] = line["cpu_baseline"].pop("oracle_verified")
    emit(line)
    if last:
        sys.stderr.write(f"[bench] last proof sha256 {hashlib.sha256(last[-1]).hexdigest()[:16]}\n")


DUMP_LIMIT_BYTES = 64_000_000  # all files of one dump, over all ranks
NPY_HEADERS_BYTES = 1024  # allowance for the headers of one rank's two .npy files


def dump_outputs(out_dir: Path, proofs: list[bytes], first_index: int, name: str, world: int, limit: int = DUMP_LIMIT_BYTES) -> None:
    """`<name>.npy`: the proofs of the last timed step, one row of 784 byte values per proof (float32, exact);
    `<name>_index.npy`: the index of each row in the step's batch (float64).  The `world` ranks share `limit` bytes
    equally; above its share a rank writes a fixed, seeded sample of its rows, so that two builds given the same
    arguments can be compared output for output."""
    import numpy as np

    rows = np.frombuffer(b"".join(proofs), dtype=np.uint8).reshape(len(proofs), 784)
    index = np.arange(len(proofs))
    keep = (limit // world - NPY_HEADERS_BYTES) // (784 * 4 + 8)
    if len(proofs) > keep:
        index = np.sort(np.random.default_rng(0).choice(len(proofs), size=keep, replace=False))
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / f"{name}.npy", rows[index].astype(np.float32))
    np.save(out_dir / f"{name}_index.npy", (index + first_index).astype(np.float64))


def workload_string(strong: bool, total: int, n_dev: int, batch: int | None) -> str:
    """`config.workload`, shared by both arms so that the driver compares like with like."""
    if strong:
        return (f"Ring VRF prove, Bandersnatch, ring {RING_SIZE} / domain 2048, one batch of {total} proofs per step sharded over {n_dev} GPU(s) "
                f"({total // n_dev} per GPU) -- BASELINE configs[1]")
    return f"Ring VRF prove, Bandersnatch, ring {RING_SIZE} / domain 2048, batch {batch} proofs per GPU per step (BASELINE configs[1] shape, weak scaling)"


def _shard(total: int, parts: int, index: int) -> tuple[int, int]:
    base, extra = divmod(total, parts)
    lo = index * base + min(index, extra)
    return lo, lo + base + (1 if index < extra else 0)


# ncu --set full captures of the dominant kernel (profiles/): dram__bytes_read.sum + dram__bytes_write.sum of ONE launch.  A 96-byte
# table entry at a random address straddles 64-byte DRAM atoms (2 or 3 of them), so the traffic exceeds the algorithmic table bytes;
# the kernel is bound by the integer pipe, not by these reads.
NCU_TRAFFIC = {
    "glv": {"bytes": 21.81e9, "launch": "CommitBodyT<true> grid (4, 1024) x 128 threads (1024 x 6145 coefficients, bench.py --total 1024), 39.8 ms under ncu: 19.91 GB read + 1.90 GB written (register spills); algorithmic table bytes of that launch 9.66e9 (profiles/r02_ncu_full_CommitBody_glv16.csv)"},
    "plain": {"bytes": 23.0e9, "launch": "CommitBody grid (2, 1024) x 128 threads, 44.6 ms under ncu; algorithmic table bytes of that launch 10.9e9 (profiles/r01_ncu_full_CommitBody_w18.csv)"},
}


# ------------------------------------------------------------------------------------ CPU baseline (oracle)
def _oracle_ring():
    from oracle import bandersnatch as bs
    from oracle import ring_proof as rp
    from oracle import transcript as tr

    pk, sk = tr.secret_from_seed(bs.SHA512, seed_bytes("batch-signer", 0, 0))
    keys = [pk if i == SIGNER_INDEX else tr.secret_from_seed(bs.SHA512, seed_bytes("ring-member", 0, i))[0] for i in range(RING_SIZE)]
    params = rp.Params.from_ring_size(RING_SIZE)
    ring = rp.Ring(keys, params)
    root = rp.RingRoot.from_ring(ring, params)
    return pk, sk, ring, root


def _oracle_prove_n(args):
    """Worker: build the ring once, then time `count` proofs."""
    count, start = args
    from oracle import fr as ofr
    from oracle import vrf as ovrf

    pk, sk, ring, root = _oracle_ring()
    rng = random.Random(start)
    t0 = time.perf_counter()
    for j in range(count):
        zk = [rng.randrange(ofr.R) for _ in range(12)]
        ovrf.ring_prove(b"bench-batch-input" + le64(start + j), b"bench-batch-ad" + le64(start + j), sk, pk, ring, root, zk_rows=zk)
    return time.perf_counter() - t0


def cpu_baseline_single(gpu_sample=()) -> dict:
    """The oracle port timed on one host core (reported baseline), and -- the checker role of the same leg -- the oracle's verifier
    run over a few proofs the GPU produced inside the timed region."""
    from oracle import backend_name

    count = int(os.environ.get("DOT_RING_B200_CPU_BASELINE_PROOFS", "10"))  # about 11 s of CPU work
    dt = _oracle_prove_n((count, 0))
    verified = 0
    if gpu_sample:
        from oracle import vrf as ovrf

        _, _, oring, oroot = _oracle_ring()
        for proof, alpha, ad in gpu_sample:
            if not ovrf.ring_verify(ovrf.RingVrfProof.decode(proof), alpha, ad, oring, oroot, ring_matches=True):
                raise SystemExit("bench.py: the CPU oracle rejects a proof of the timed region; refusing to report a number")
            verified += 1
    return {
        "oracle_verified": verified,
        "value": count / dt,
        "unit": "proofs/s",
        "cores": 1,
        "kind": "port",
        "sample": f"{count} proofs, ring {RING_SIZE} / domain 2048, oracle port ({backend_name()}), ring set-up excluded",
    }


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from concurrent.futures import ProcessPoolExecutor

    from oracle import backend_name

    cores = os.cpu_count() or 1
    workers = max(1, min(cores, args.ref_workers or cores))
    total_steps = args.steps + args.warmup
    with ProcessPoolExecutor(max_workers=workers) as ex:
        times = list(ex.map(_oracle_prove_n, [(total_steps, 1000 * w) for w in range(workers)]))
    # every worker proves one proof per step; warm-up steps are part of each worker's loop, so scale them out
    per_worker_s = [t * args.steps / total_steps for t in times]
    wall = max(per_worker_s)
    value = workers * args.steps / wall
    line = {
        "impl": "reference",
        "impl_note": "PORT: the CPU oracle's restatement of the reference's algorithm (Python + a plain-C Pippenger), one process per host core; the reference's own package "
                     "cannot be built offline (its setup.py clones blst).  Its published native-blst figure is ~2x this port per core (docs/BENCHMARK.md:72: 1.9 proofs/s on an M1 Max core).",
        "metric": "ring_vrf_proofs_per_s",
        "value": value,
        "unit": "proofs/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": wall * 1e3 / args.steps,
        "higher_is_better": True,
        "scaling": args.scaling,
        "vs_baseline": None,
        "dtype": "python ints / u64 limbs",
        "data": "synthetic",
        "config": {"workload": workload_string(args.scaling == "strong", args.total, args.gpus, args.batch),
                   "sample": f"bounded sample of that workload: each step = 1 proof on each of {workers} host processes (the CPU path has no batch dimension: its rate does not depend on the batch size)"},
        "cpu_baseline": {"value": value, "unit": "proofs/s", "cores": workers, "kind": "port", "sample": f"{workers} x {args.steps} proofs, oracle port ({backend_name()}): the reference's algorithm restated (its own package cannot be built offline, DESIGN.md section 7)"},
        "e2e": {"value": value, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line goes to the process's original stdout; everything else (NCCL banners, library chatter) was
    re-routed to stderr in main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main() -> None:
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # fd 1 -> stderr for native libraries (NCCL prints its version banner on stdout)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default, BASELINE configs[1]): one batch of --total proofs per step sharded over the GPUs; weak: --batch proofs per GPU per step")
    ap.add_argument("--total", type=int, default=4096, help="proofs per step over all GPUs (strong scaling)")
    ap.add_argument("--batch", type=int, default=None, help="proofs per GPU per step; giving it selects --scaling weak (8192 = one full-width device pass)")
    ap.add_argument("--saturated-batch", type=int, default=8192, help="also report the saturated operating point: this many proofs per GPU per step (0 = skip)")
    ap.add_argument("--saturated-steps", type=int, default=3)
    ap.add_argument("--window-bits", type=int, default=int(os.environ.get("DOT_RING_B200_WINDOW_BITS", "16")),
                    help="fixed-base table window width; 0 = sized by the library. Default: 16-bit windows over GLV halves (16 additions per coefficient, 161 GB); "
                    "if that does not fit the run falls back to 14-bit windows with four 15-bit ones (18 additions, 106 GB)")
    ap.add_argument("--wide-windows", type=int, default=None, help="how many low windows take one more bit (default 4 with 14-bit windows)")
    ap.add_argument("--glv", type=int, default=None, help="1: table over 128 bits, scalars split with the G1 endomorphism (2 x windows additions per coefficient)")
    ap.add_argument("--prove-chunk", type=int, default=int(os.environ.get("DOT_RING_B200_PROVE_CHUNK", "0")), help="proofs per device pass (0: the library's choice, at most 4096)")
    ap.add_argument("--commit-mode", type=int, default=int(os.environ.get("DOT_RING_B200_COMMIT_MODE", "0")), help="0 XYZZ accumulation, 1 batched-affine rounds")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-workers", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the proofs of the last timed step to DIR/proofs.npy (float32 byte values, one row per proof) and their batch indices to DIR/proofs_index.npy; "
                    "inside the repository use bench_outputs/, which git ignores")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the proofs of this engine; --impl reference keeps none")
    if args.batch is not None:
        args.scaling = "weak"
    elif args.scaling == "weak":
        args.batch = 8192
    if args.glv is None:
        args.glv = int(os.environ.get("DOT_RING_B200_GLV", "1" if args.window_bits == 16 else "0"))
    if args.wide_windows is None:
        args.wide_windows = int(os.environ.get("DOT_RING_B200_WIDE_WINDOWS", "4" if args.window_bits == 14 and not args.glv else "0"))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
