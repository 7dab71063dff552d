"""Ring and RingRoot: drop-in mirrors of dot_ring/vrf/ring/members.py:18-81 and dot_ring/vrf/ring/root.py:13-112.

``Ring(keys, params)`` ingests the keys on the GPU (batched decompression + prime-subgroup check,
invalid keys -> padding point), builds the public vector ``PK || padding || 2^i*B || zeros`` and, in the
same device object, the three fixed columns (px, py, s): coefficients, KZG commitments (= the ring
root) and their 4x low-degree extensions.  The reference recomputes the latter on every proof
(constraints.py:43-62); here they live in HBM for the lifetime of the ring.

``RingVerifier(roots)`` verifies Ring VRF proofs against ring roots alone: the verifier needs neither the keys nor the SRS
window table, and one batch may span several rings (one aggregated pairing check for all of them).

``RingRoot.from_keys(keys, params)`` derives a root from keys without a ``Ring`` or that table, and ``root.update(rows, new_keys,
old_keys)`` follows a change of a few rows from the root alone (the root is linear in the column evaluations).
"""

from __future__ import annotations

from collections.abc import Sequence
from dataclasses import dataclass, field
from functools import lru_cache
from typing import Any

from . import _native
from .curve import point_to_string
from .engine import Engine, EnginePool, PooledRingNative, default_engine
from .params import RingProofParams


def _native_ring(engine: Engine, keys: Sequence[bytes], params: RingProofParams) -> _native.NativeRing:
    p = params.cv.curve.params
    aux = p.auxiliary_points
    return _native.NativeRing(
        engine.srs,
        [bytes(k) for k in keys],
        domain_size=params.domain_size,
        max_ring_size=params.max_ring_size,
        padding_rows=params.padding_rows,
        omega=params.omega,
        radix_omega=params.radix_omega,
        seed=aux.accumulator_base,
        blinding_base=aux.blinding_base,
        padding_point=aux.padding_point,
        generator=p.generator,
        suite_id=p.suite_id,
        h2c_dst=p.hash_to_curve.dst,
        hash_name=p.hash_name,
    )


class Ring:
    nm_points: tuple[tuple[int, int], ...]
    params: RingProofParams

    def __init__(self, keys: Sequence[bytes], params: RingProofParams | None = None, engine: "Engine | EnginePool | None" = None) -> None:
        if params is None:
            params = RingProofParams.from_ring_size(len(keys))
        self.params = params
        self.engine = engine or default_engine()
        aux = params.cv.curve.params.auxiliary_points
        if not aux.padding_point:
            raise ValueError("padding point is not configured in curve parameters")
        if len(keys) > params.max_ring_size:
            raise ValueError(f"ring size {len(keys)} exceeds max supported size {params.max_ring_size}")
        self.keys = tuple(bytes(k) for k in keys)
        # keys of the wrong length can never decode; the reference maps them to the padding point as well
        normalised = [k if len(k) == 32 else b"\xff" * 32 for k in self.keys]
        if isinstance(self.engine, EnginePool):  # one replica per GPU; batches are sharded over them (engine.py)
            self.native = PooledRingNative(self.engine, lambda eng: _native_ring(eng, normalised, params))
        else:
            self.native = _native_ring(self.engine, normalised, params)
        self.nm_points = tuple(self.native.points())
        self._index: dict[tuple[int, int], int] | None = None

    @classmethod
    def from_keys(cls, keys: Sequence[bytes], params: RingProofParams | None = None) -> "Ring":
        """Cached ring for a stable encoded key vector (members.py:57-59)."""
        return _ring(tuple(bytes(key) for key in keys))

    def _decode_key(self, key: bytes) -> tuple[int, int] | None:
        if len(key) != 32:
            return None
        pt = self.engine.ctx.te_decode([bytes(key)], checked=True)[0]
        if pt is None or pt == (0, 1):
            return None
        return pt

    def index_of(self, key: bytes) -> int:
        """members.py:71-81."""
        padding_point = self.params.cv.curve.params.auxiliary_points.padding_point
        point = self._decode_key(key)
        if point is None:
            raise ValueError("invalid ring key")
        if point == padding_point:
            raise ValueError("producer key is not in ring")
        if self._index is None:
            index: dict[tuple[int, int], int] = {}
            for i, pt in enumerate(self.nm_points[: self.params.max_ring_size]):
                index.setdefault(pt, i)
            self._index = index
        try:
            return self._index[point]
        except KeyError as exc:
            raise ValueError("producer key is not in ring") from exc


@lru_cache(maxsize=2)
def _params(keys_len: int) -> RingProofParams:
    return RingProofParams.from_ring_size(keys_len)


@lru_cache(maxsize=8)
def _ring(keys: tuple[bytes, ...]) -> Ring:
    return Ring(keys, _params(len(keys)))


@dataclass
class Column:
    """Commitment holder mirroring dot_ring/ring_proof/columns/columns.py:21-60 (device keeps evals/coeffs)."""

    name: str
    _commitment: bytes | None = None
    size: int = 512

    @property
    def commitment(self) -> bytes:
        if self._commitment is None:
            raise ValueError(f"{self.name} commitment is not set")
        return self._commitment


def _run_on(engine: "Engine | EnginePool | None", fn):
    """fn(engine) (None: the default engine); for a pool, fn(its first engine) on that engine's worker thread: a root is a few
    hundred thousand additions, not worth sharding."""
    engine = engine or default_engine()
    if isinstance(engine, EnginePool):
        return engine.map(lambda i: fn(engine.engines[i]), [0])[0]
    return fn(engine)


def _root_params(params: RingProofParams) -> _native.RingParamsStruct:
    """The dr_ring_params of `params` as the root functions read them."""
    aux = params.cv.curve.params.auxiliary_points
    if not aux.padding_point:
        raise ValueError("padding point is not configured in curve parameters")
    return _native.make_ring_params(domain_size=params.domain_size, max_ring_size=params.max_ring_size, padding_rows=params.padding_rows, omega=params.omega,
                                    seed=aux.accumulator_base, blinding_base=aux.blinding_base, padding_point=aux.padding_point, generator=(0, 0), suite_id=b"",
                                    h2c_dst=b"")  # fmt: skip


def _ring_keys(keys: Sequence[bytes]) -> list[bytes]:
    """Keys of the wrong length can never decode: as in Ring, they become keys that map to the padding point."""
    return [bytes(k) if len(k) == 32 else b"\xff" * 32 for k in keys]


@dataclass
class RingRoot:
    px: Column
    py: Column
    s: Column
    params: RingProofParams | None = None
    engine: Any = field(default=None, compare=False, repr=False)  # what `update` commits with (None: the default engine)

    @classmethod
    def _from_bytes(cls, data: bytes, params: RingProofParams, eng: Engine, owner) -> "RingRoot":
        pts, _ = eng.ctx.g1_decompress(data)
        n = params.domain_size
        return cls(px=Column("px", pts[0:96], n), py=Column("py", pts[96:192], n), s=Column("s", pts[192:288], n), params=params, engine=owner)

    @classmethod
    def from_keys(cls, keys: Sequence[bytes], params: RingProofParams | None = None, engine: "Engine | EnginePool | None" = None) -> "RingRoot":
        """`RingRoot.from_ring(Ring(keys, params))` without the ring: the keys' public vector committed on the device with the
        engine's small root table (`Engine.root_srs`), never the prover's window table."""
        if params is None:
            params = RingProofParams.from_ring_size(len(keys))
        return cls.from_key_sets([keys], params, engine)[0]

    @classmethod
    def from_key_sets(cls, key_sets: Sequence[Sequence[bytes]], params: RingProofParams, engine: "Engine | EnginePool | None" = None) -> list["RingRoot"]:
        """`from_keys` of every key set under one params, in one device call."""
        sets = [_ring_keys(keys) for keys in key_sets]
        for keys in sets:
            if len(keys) > params.max_ring_size:
                raise ValueError(f"ring size {len(keys)} exceeds max supported size {params.max_ring_size}")
        struct = _root_params(params)

        def run(eng: Engine):
            roots = _native.ring_roots_from_keys(eng.root_srs(params.domain_size), struct, sets)
            return [cls._from_bytes(r, params, eng, engine) for r in roots]

        return _run_on(engine, run)

    def update(self, rows: Sequence[int], new_keys: Sequence[bytes], old_keys: Sequence[bytes] | None = None) -> "RingRoot":
        """The root after row rows[j] went from old_keys[j] to new_keys[j] (old_keys None: the rows held padding, an append); a
        new key that does not decode nulls its row.  Needs only this root, not the other keys; `self` is left as it is."""
        if self.params is None:
            raise ValueError("updating a ring root requires its ring proof parameters")
        params = self.params
        struct = _root_params(params)
        new = _ring_keys(new_keys)
        old = None if old_keys is None else _ring_keys(old_keys)

        def run(eng: Engine):
            data = eng.ctx.g1_compress(b"".join(self.fixed_commitments()))
            out = _native.ring_root_update(eng.root_srs(params.domain_size), struct, data, list(rows), new, old)
            return RingRoot._from_bytes(out, params, eng, self.engine)

        return _run_on(self.engine, run)

    @classmethod
    def from_ring(cls, ring: Ring, params: RingProofParams | None = None) -> "RingRoot":
        """root.py:21-44: the three commitments were produced when the ring was ingested."""
        if params is None:
            params = ring.params
        if (params.domain_size, params.max_ring_size) != (ring.params.domain_size, ring.params.max_ring_size):
            ring = Ring(ring.keys, params, ring.engine)
        raw = ring.native.fixed_commitments()
        n = params.domain_size
        return cls(
            px=Column("px", raw[0:96], n), py=Column("py", raw[96:192], n), s=Column("s", raw[192:288], n), params=params
        )

    def fixed_commitments(self) -> list[Any]:
        return [self.px.commitment, self.py.commitment, self.s.commitment]

    def verifier_transcript_prefix(self, transcript_challenge: bytes | None = None):
        """root.py:54-71: transcript state after absorbing the verifier key = [1]_1 | [1]_2 | [tau]_2 | C_px | C_py | C_s (uncompressed)."""
        if self.params is None:
            raise ValueError("Ring root verifier transcript requires ring proof parameters")
        from .transcript import FiatShamirTranscript

        srs = default_engine().srs_bytes
        if transcript_challenge is None:
            transcript_challenge = self.params.cv.curve.params.suite_id
        transcript = FiatShamirTranscript(self.params.prime, transcript_challenge)
        transcript.absorb_labeled(b"vk", srs.g1_be96[:96] + srs.g2_be192 + b"".join(self.fixed_commitments()))
        return transcript

    @staticmethod
    def encoded_len(params: RingProofParams | None = None) -> int:
        return 3 * 48

    def encode(self) -> bytes:
        from .kzg import KZG

        pcs = self.params.pcs if self.params is not None else KZG
        return pcs.compress_g1(self.px.commitment + self.py.commitment + self.s.commitment)

    @classmethod
    def decode(cls, data: bytes, ring: Ring | RingProofParams | None = None) -> "RingRoot":
        """root.py:89-109."""
        params = ring.params if isinstance(ring, Ring) else ring
        if params is None:
            params = RingProofParams()
        expected = cls.encoded_len(params)
        if len(data) != expected:
            raise ValueError(f"invalid ring root length: ring root must be exactly {expected} bytes, got {len(data)}")
        pts = params.pcs.decompress_g1_batch(bytes(data))
        n = params.domain_size
        return cls(px=Column("px", pts[0], n), py=Column("py", pts[1], n), s=Column("s", pts[2], n), params=params)

    def matches_ring(self, ring: Ring) -> bool:
        """root.py:111-112."""
        return RingRoot.from_ring(ring).encode() == self.encode()


def _suite_key(params: RingProofParams):
    p = params.cv.curve.params
    return (p.suite_id, p.hash_to_curve.dst, p.hash_name, tuple(p.generator), tuple(p.auxiliary_points.blinding_base))


def _native_verifier(engine: Engine, root: bytes, params: RingProofParams) -> _native.NativeRingVerifier:
    p = params.cv.curve.params
    srs = engine.srs_bytes  # [1]_1 and the G2 points only: the window table (`engine.srs`) is never built here
    return _native.NativeRingVerifier(
        engine.ctx, root, srs.g1_be96[:96], srs.g2_be192, domain_size=params.domain_size, omega=params.omega, seed=p.auxiliary_points.accumulator_base,
        blinding_base=p.auxiliary_points.blinding_base, generator=p.generator, suite_id=p.suite_id, h2c_dst=p.hash_to_curve.dst, hash_name=p.hash_name,
    )  # fmt: skip


class RingVerifier:
    """Ring VRF verification against ring roots alone (the verifier side of vrf/ring/vrf.py:226-283 without the ``Ring``).

    ``roots`` are :class:`RingRoot` values (``RingRoot.decode(data, params)`` or ``RingRoot.from_ring(ring)``), each with its
    ``params``; they must share the suite, their domain sizes may differ.  Item i of a batch is checked against
    ``roots[rings[i]]`` (default: every item against ``roots[0]``).  ``batch_verify`` folds the whole batch, whatever the
    ring of each item, into one pairing check.  With an :class:`EnginePool` every device holds one verifier per root and takes a
    contiguous shard of the batch; the aggregated result is then the conjunction of the devices' checks."""

    def __init__(self, roots: Sequence[RingRoot], engine: "Engine | EnginePool | None" = None) -> None:
        roots = list(roots)
        if not roots:
            raise ValueError("RingVerifier needs at least one ring root")
        if any(r.params is None for r in roots):
            raise ValueError("every ring root must carry its ring proof parameters")
        if len({_suite_key(r.params) for r in roots}) != 1:
            raise ValueError("ring roots of one RingVerifier must share the suite")
        self.roots = roots
        self.params = roots[0].params
        self.engine = engine or default_engine()
        encoded = [r.encode() for r in roots]

        def build(eng: Engine):
            out = []
            try:
                for data, r in zip(encoded, roots):
                    out.append(_native_verifier(eng, data, r.params))
            except BaseException:
                for v in out:
                    v.close()
                raise
            return out

        if isinstance(self.engine, EnginePool):
            self.replicas = self.engine.map(lambda i: build(self.engine.engines[i]))
        else:
            self.replicas = [build(self.engine)]

    def close(self) -> None:
        for verifiers in self.replicas:
            for v in verifiers:
                v.close()
        self.replicas = []

    def _verify_common(self, proofs, inputs, additional_data, rings, aggregate: bool):
        """-> (per-item verdicts, all_ok); coefficients drawn as in RingVRF._verify_common."""
        from .kzg import _random_nonzero_coefficients

        raw = [bytes(p) if isinstance(p, (bytes, bytearray)) else p.encode() for p in proofs]
        n = len(raw)
        if not (len(inputs) == len(additional_data) == n):
            raise ValueError("proofs, inputs and additional_data must have the same length")
        index = [0] * n if rings is None else [int(k) for k in rings]
        if len(index) != n:
            raise ValueError("rings must give one ring index per proof")
        if any(not 0 <= k < len(self.roots) for k in index):
            raise ValueError("ring index out of range")
        if n == 0:
            return [], True
        order = self.params.prime
        if aggregate:
            coeffs = _random_nonzero_coefficients(2 * n, order)
        else:  # independent checks: (1, r) per proof
            coeffs = [v for r in _random_nonzero_coefficients(n + 1, order)[1:] for v in (1, r)]
        inputs = [bytes(a) for a in inputs]
        ads = [bytes(d) for d in additional_data]
        bounds = EnginePool.shard_bounds(n, len(self.replicas))

        def run(i):
            lo, hi = bounds[i]
            return _native.NativeRingVerifier.verify_multi(self.replicas[i], index[lo:hi], inputs[lo:hi], ads[lo:hi], raw[lo:hi], coeffs[2 * lo : 2 * hi], aggregate)

        if len(bounds) <= 1:
            return run(0)
        parts = self.engine.map(run, range(len(bounds)))
        return [v for verdicts, _ in parts for v in verdicts], all(ok for _, ok in parts)

    def verify(self, proof, input: bytes, ad: bytes, ring: int = 0) -> bool:
        """vrf/ring/vrf.py:226-232 against roots[ring]."""
        return self._verify_common([proof], [input], [ad], [ring], False)[0][0] == 1

    def verify_batch(self, proofs, inputs, additional_data, rings: Sequence[int] | None = None) -> list[int]:
        """Independent verifications, item i against roots[rings[i]]: 1 valid, 0 invalid, 2 malformed encoding."""
        return self._verify_common(proofs, inputs, additional_data, rings, False)[0]

    def batch_verify(self, proofs, inputs, additional_data, rings: Sequence[int] | None = None) -> bool:
        """vrf/ring/vrf.py:239-283 over a batch that may span all the roots: one pairing check (one per device of a pool);
        any error -> False."""
        try:
            return self._verify_common(proofs, inputs, additional_data, rings, True)[1]
        except (AssertionError, AttributeError, TypeError, ValueError):
            return False


__all__ = ["Ring", "RingRoot", "RingVerifier", "Column", "point_to_string"]
