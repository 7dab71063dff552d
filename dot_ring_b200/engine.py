"""Process-wide engine: one CUDA context + SRS (with its fixed-base table) per GPU.

The reference keeps a module-level ``KZG.srs`` (dot_ring/ring_proof/pcs/kzg.py:114-119); the
equivalent here is a lazily created :class:`Engine` per device, holding the ``dr_ctx`` and ``dr_srs``
handles.  Device selection is a property of the engine (``DOT_RING_B200_DEVICE`` or
``Engine(device=...)``), not of ``RingProofParams``.
"""

from __future__ import annotations

import os
import threading

from . import _native
from .srs import SrsBytes, read_srs_file

_lock = threading.Lock()
_engines: dict[int, "Engine"] = {}


class Engine:
    def __init__(self, device: int = 0, window_bits: int | None = None, library: _native.Library | None = None, srs_points: int | None = None,
                 srs: "SrsBytes | None" = None, wide_windows: int = 0, glv: bool = False):
        self.device = device
        self.ctx = _native.Context(device, library)
        env = os.environ.get("DOT_RING_B200_WINDOW_BITS")
        # None / 0 = let the library size the table from the free HBM (dr_srs_load); wide_windows only with an explicit width
        self.window_bits = int(window_bits) if window_bits is not None else (int(env) if env else 0)
        self.wide_windows = int(wide_windows) if self.window_bits else 0
        self.glv = bool(glv) if self.window_bits else False
        self._srs: _native.NativeSrs | None = None
        self._root_srs: dict[int, _native.NativeSrs] = {}
        self._srs_points = srs_points
        # `srs` overrides the bundled 6145-point file (needed for domains above 2048, whose quotient has 3N + 1 coefficients)
        self.srs_bytes = srs if srs is not None else read_srs_file(None, srs_points)

    @property
    def srs(self) -> _native.NativeSrs:
        """SRS points + window table in HBM, built on first use (about 3.5 s for the 106 GB table a B200 gets by default)."""
        if self._srs is None:
            self._srs = _native.NativeSrs(self.ctx, self.srs_bytes.g1_be96, self.srs_bytes.g2_be192, self.window_bits, self.wide_windows, self.glv)
            self.window_bits, self.wide_windows, glv, self.table_additions = self._srs.geometry
            self.glv = bool(glv)
        return self._srs

    def root_srs(self, domain_size: int) -> _native.NativeSrs:
        """The first `domain_size` SRS points with a small fixed-base table, built on first use per domain size: ring roots are
        committed with it (`RingRoot.from_keys`, `RingRoot.update`), so deriving a root never builds the prover's table (`srs`).
        4-bit windows over the GLV halves: 64 table additions per coefficient, 24.6 KB per point (50 MB at N = 2048, 1.6 GB at
        N = 65536); a root is a few hundred thousand additions."""
        srs = self._root_srs.get(domain_size)
        if srs is None:
            srs = _native.NativeSrs(self.ctx, self.srs_bytes.g1_be96[: 96 * domain_size], self.srs_bytes.g2_be192, 4, 0, True)
            self._root_srs[domain_size] = srs
        return srs

    def close(self) -> None:
        if self._srs is not None:
            self._srs.close()
            self._srs = None
        for srs in self._root_srs.values():
            srs.close()
        self._root_srs.clear()
        self.ctx.close()


def default_engine() -> Engine:
    """The engine behind the module-level API (``KZG``, ``TinyVRF`` ...): what `set_default_engine` installed (an
    :class:`Engine` or an :class:`EnginePool`), else a lazily created single-device engine."""
    device = int(os.environ.get("DOT_RING_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    with _lock:
        eng = _engines.get(device)
        if eng is None:
            eng = Engine(device)
            _engines[device] = eng
        return eng


def set_default_engine(engine: Engine | None, device: int = 0) -> None:
    """Install (or drop) the engine used by the module-level API; tests use it to inject the emulation build."""
    with _lock:
        if engine is None:
            _engines.pop(device, None)
        else:
            _engines[device] = engine


class EnginePool:
    """One :class:`Engine` (``dr_ctx`` + SRS window table + ring replicas) per GPU of the node, behind one Python process.

    The path shards naturally (SURVEY.md 8e): proofs and verifications are independent units, so a caller's batch is split
    into contiguous shards, one per device, and the results are concatenated in order; nothing is exchanged between GPUs.
    Every device has its own worker thread; ctypes releases the GIL for the duration of a C-ABI call, so the shards run
    concurrently.  This is what the reference does with a process pool over one work list
    (tests/benchmark/bench_ring_proof.py:168-182).

    ``Ring(keys, params, engine=pool)`` builds one ring replica per device (in parallel) and
    ``RingVRF.prove_batch`` / ``verify_batch`` / ``batch_verify`` then use every GPU of the pool.
    """

    def __init__(self, devices=None, **engine_kwargs):
        from concurrent.futures import ThreadPoolExecutor

        if devices is None:
            devices = range(_native.default_library().device_count())
        self.devices = [int(d) for d in devices]
        if not self.devices:
            raise ValueError("EnginePool needs at least one device")
        self._workers = [ThreadPoolExecutor(max_workers=1, thread_name_prefix=f"dr-gpu{d}") for d in self.devices]
        self.engines = self.map(lambda i: Engine(self.devices[i], **engine_kwargs))
        self.ctx = PooledContext(self)
        self.srs_bytes = self.engines[0].srs_bytes

    def __len__(self) -> int:
        return len(self.engines)

    @property
    def srs(self):
        """First device's SRS (all replicas are built on demand by ``warm``)."""
        return self.engines[0].srs

    def map(self, fn, indices=None) -> list:
        """Run ``fn(i)`` on worker i for every i in `indices` (default: all) concurrently; results in index order."""
        idx = list(range(len(self._workers))) if indices is None else list(indices)
        futures = [self._workers[i].submit(fn, i) for i in idx]
        return [f.result() for f in futures]

    def warm(self) -> None:
        """Build every device's window table now (concurrently) instead of at the first commitment."""
        self.map(lambda i: self.engines[i].srs)

    def g1_msm(self, points_be96: bytes, scalars, min_points_per_device: int = 1 << 16) -> bytes:
        """`KZG.msm_g1` split by POINT RANGE over the devices (BASELINE north star: "large MSMs split by point range, partial G1
        sums combined on the host"): device i computes sum_{j in range i} k_j P_j, the partial sums (96 bytes each) come back to
        the host and are added by one more, tiny, MSM with unit scalars.  Only worth it for very large sets: every device pays
        the bucket method's latency floor (~2 ms) and the combine another, so ranges shorter than `min_points_per_device` are
        not split (measured in round 1 at 196 609 points: 11 ms on one GPU, 42 ms split over eight)."""
        n = len(points_be96) // 96
        if isinstance(scalars, (bytes, bytearray)):
            ks = bytes(scalars)
        else:
            ks = b"".join((int(k) % _native.FR_MODULUS).to_bytes(32, "little") for k in scalars)
        if len(ks) != 32 * n:
            raise ValueError("points and scalars must have the same length")
        parts = max(1, min(len(self), n // max(1, min_points_per_device)))
        bounds = self.shard_bounds(n, parts)
        if len(bounds) <= 1:
            return self.engines[0].ctx.g1_msm(points_be96, ks)
        partial = self.map(lambda i: self.engines[i].ctx.g1_msm(points_be96[96 * bounds[i][0] : 96 * bounds[i][1]], ks[32 * bounds[i][0] : 32 * bounds[i][1]]), range(len(bounds)))
        return self.engines[0].ctx.g1_msm(b"".join(partial), [1] * len(partial))

    @staticmethod
    def shard_bounds(n: int, parts: int) -> list[tuple[int, int]]:
        """Contiguous, balanced shards: the first n % parts shards take one extra item; empty shards are dropped."""
        base, extra = divmod(n, parts)
        out, lo = [], 0
        for i in range(parts):
            hi = lo + base + (1 if i < extra else 0)
            if hi > lo:
                out.append((lo, hi))
            lo = hi
        return out

    def close(self) -> None:
        self.map(lambda i: self.engines[i].close())
        for w in self._workers:
            w.shutdown(wait=True)


class PooledContext:
    """``_native.Context`` interface over a pool: the batched Tiny / Thin / Pedersen calls (independent items, lists in the
    same order as the reference's per-item API) are sharded contiguously over the devices; everything else (single-item
    helpers, codecs, settings) goes to the first device."""

    _SHARDED = {"pedersen_verify": 1, "thin_verify": 1, "tiny_verify": 1, "vrf_prove": 2, "pedersen_prove_with_blinding": 1}  # index of the first list argument
    _MIN_ITEMS_PER_DEVICE = 256

    def __init__(self, pool: "EnginePool"):
        self._pool = pool

    def __getattr__(self, name):
        first = self._pool.engines[0].ctx
        attr = getattr(first, name)
        if name not in self._SHARDED:
            return attr
        lead = self._SHARDED[name]
        pool = self._pool

        def sharded(*args, **kwargs):
            n = len(args[lead])
            parts = max(1, min(len(pool), n // self._MIN_ITEMS_PER_DEVICE))
            bounds = pool.shard_bounds(n, parts)
            if len(bounds) <= 1:
                return attr(*args, **kwargs)

            def run(i):
                lo, hi = bounds[i]
                sliced = [a[lo:hi] if j >= lead and isinstance(a, (list, tuple)) and len(a) == n else a for j, a in enumerate(args)]
                return getattr(pool.engines[i].ctx, name)(*sliced, **kwargs)

            out = pool.map(run, range(len(bounds)))
            if isinstance(out[0], tuple):  # (proofs, blinding factors)
                return tuple([x for part in out for x in part[k]] for k in range(len(out[0])))
            return [x for part in out for x in part]

        return sharded


class PooledRingNative:
    """The ``NativeRing`` interface over one replica per device of an :class:`EnginePool` (same results, sharded batches)."""

    def __init__(self, pool: EnginePool, make_replica):
        self.pool = pool
        self.replicas = pool.map(lambda i: make_replica(pool.engines[i]))
        self.ctx = self.replicas[0].ctx
        self.domain_size = self.replicas[0].domain_size

    def close(self) -> None:
        self.pool.map(lambda i: self.replicas[i].close())

    @property
    def time_calls(self) -> bool:
        return self.replicas[0].time_calls

    @time_calls.setter
    def time_calls(self, on: bool) -> None:
        for r in self.replicas:
            r.time_calls = bool(on)

    @property
    def last_call_ms(self) -> float:
        """Device time of the slowest replica's last prove call."""
        return max(r.last_call_ms for r in self.replicas)

    def root(self) -> bytes:
        return self.replicas[0].root()

    def fixed_commitments(self) -> bytes:
        return self.replicas[0].fixed_commitments()

    def points(self):
        return self.replicas[0].points()

    def witness_table_bits(self) -> int:
        return self.replicas[0].witness_table_bits()

    def commit_kernel_ms(self) -> tuple[float, int]:
        per = self.pool.map(lambda i: self.replicas[i].commit_kernel_ms())
        return max(per)

    def prove_phase_ms(self) -> list[float]:
        """Per-phase device time of the slowest replica's last call."""
        per = self.pool.map(lambda i: self.replicas[i].prove_phase_ms())
        return max(per, key=sum)

    def prove_batch(self, alphas, ads, secret_keys, producer_index, zk_rows=None):
        """The batch is packed ONCE on the calling thread (the packing holds the GIL: done per shard it would serialise the
        workers); every device then proves a contiguous sub-range of the same flat buffers and writes its proofs into its slice
        of one output buffer."""
        n = len(alphas)
        bounds = self.pool.shard_bounds(n, len(self.replicas))
        if len(bounds) <= 1:
            return self.replicas[0].prove_batch(alphas, ads, secret_keys, producer_index, zk_rows)
        pk = _native.NativeRing.pack_prove_inputs(alphas, ads, secret_keys, producer_index, zk_rows)
        self.pool.map(lambda i: self.replicas[i].prove_packed(pk, bounds[i][0], bounds[i][1]), range(len(bounds)))
        return _native.NativeRing.unpack_proofs(pk)

    @staticmethod
    def prove_multi(rings: list["PooledRingNative"], index, alphas, ads, secret_keys, producer_index, zk_rows=None):
        """Item i against rings[index[i]] (`NativeRing.prove_multi`): the batch is packed once and sharded contiguously; device d
        proves its shard against its own replicas of the rings.  Every ring must be built on the same pool."""
        if not rings:
            if len(alphas):
                raise ValueError("at least one ring is required")
            return [], []
        pool = rings[0].pool
        if any(not isinstance(r, PooledRingNative) or r.pool is not pool for r in rings):
            raise ValueError("rings of one call must be built on the same EnginePool")
        pk = _native.NativeRing.pack_prove_inputs(alphas, ads, secret_keys, producer_index, zk_rows, ring_index=index)
        bounds = pool.shard_bounds(pk["n"], len(pool))
        pool.map(lambda i: _native.NativeRing.prove_multi_packed([r.replicas[i] for r in rings], pk, bounds[i][0], bounds[i][1]), range(len(bounds)))
        return _native.NativeRing.unpack_proofs(pk)

    @staticmethod
    def proof_prove_multi(rings: list["PooledRingNative"], index, producer_index, blindings, zk_rows=None, label=None):
        """Bare ring proofs (`NativeRing.proof_prove_multi`) sharded as `prove_multi`: packed once, device d proves a contiguous shard
        against its own replicas of the rings."""
        if not rings:
            if len(index):
                raise ValueError("at least one ring is required")
            return [], []
        pool = rings[0].pool
        if any(not isinstance(r, PooledRingNative) or r.pool is not pool for r in rings):
            raise ValueError("rings of one call must be built on the same EnginePool")
        pk = _native.NativeRing.pack_ring_proof_inputs(index, producer_index, blindings, zk_rows, label)
        bounds = pool.shard_bounds(pk["n"], len(pool))
        pool.map(lambda i: _native.NativeRing.proof_prove_multi_packed([r.replicas[i] for r in rings], pk, bounds[i][0], bounds[i][1]), range(len(bounds)))
        return _native.NativeRing.unpack_ring_proofs(pk)

    def verify_batch(self, inputs, ads, proofs, coeffs, aggregate: bool = False):
        """Per-item mode: shards are independent.  Aggregated mode (`RingVRF.batch_verify`): every device folds its shard into
        its own random-linear-combination check (its slice of the caller's coefficients) and the batch is accepted iff every
        shard is -- the conjunction of independent batch checks, run concurrently, instead of shipping partial sums to one GPU."""
        n = len(proofs)
        bounds = self.pool.shard_bounds(n, len(self.replicas))
        if len(bounds) <= 1:
            return self.replicas[0].verify_batch(inputs, ads, proofs, coeffs, aggregate)
        parts = self.pool.map(
            lambda i: self.replicas[i].verify_batch(inputs[bounds[i][0] : bounds[i][1]], ads[bounds[i][0] : bounds[i][1]], proofs[bounds[i][0] : bounds[i][1]],
                                                    coeffs[2 * bounds[i][0] : 2 * bounds[i][1]], aggregate),
            range(len(bounds)),
        )
        return [v for verdicts, _ in parts for v in verdicts], all(ok for _, ok in parts)
