"""RingProof: the ring proof alone, `RingProofBuilder(...).build()` (dot_ring/ring_proof/proof_builder.py:38-142) batched over items.

A Ring VRF proof is a Pedersen VRF proof (which fixes the blinding factor t) next to a ring proof that ``relation = PK_k + t * B`` for
some ring row k.  ``RingProof`` offers the second half on its own: the caller brings t (for example
``PedersenVRF.prove_batch(...)[i]._blinding_factor``, or a fresh one for a plain anonymous-membership proof) and may choose the
transcript label (default: the suite id; ``b"w3f-ring-proof-test"`` for w3f ring-proof verifiers).  ``RingProof.verify_batch``
checks such proofs against a ring root alone.
"""

from __future__ import annotations

from collections.abc import Sequence
from dataclasses import dataclass

from . import _native
from .engine import EnginePool, PooledRingNative, default_engine
from .ring import Ring, RingRoot
from .vrf import _blinding_rows

RING_PAYLOAD_LEN = 592


@dataclass(frozen=True)
class RingProof:
    relation: tuple[int, int]  # PK_k + t * B, affine
    payload: bytes  # proof_payload.py:68-91

    def encode(self) -> bytes:
        return self.payload

    @classmethod
    def prove_batch(cls, ring: Ring, producer_keys: Sequence[bytes], blindings: Sequence[int], zk_rows=None, transcript_label: bytes | None = None) -> list["RingProof"]:
        """Item i proves that ``producer_keys[i]`` is in ``ring``, re-randomised by ``blindings[i]``, in one device pass."""
        return cls.prove_multi([ring], [0] * len(producer_keys), producer_keys, blindings, zk_rows, transcript_label)

    @classmethod
    def prove_multi(cls, rings: Sequence[Ring], ring_index: Sequence[int], producer_keys: Sequence[bytes], blindings: Sequence[int], zk_rows=None,
                    transcript_label: bytes | None = None) -> list["RingProof"]:
        """Item i against ``rings[ring_index[i]]``, every ring in one device pass (rings as in ``RingVRF.prove_multi``: one suite, one
        engine or one EnginePool, any domain sizes).  Keys are mapped with ``Ring.index_of`` (ValueError when absent).  Blinding rows
        as in ``RingVRF.prove_batch``: zeros for rings with ``test_vectors=True``, else ``zk_rows`` or fresh draws."""
        rings = list(rings)
        index = [int(k) for k in ring_index]
        n = len(index)
        if not (len(producer_keys) == len(blindings) == n):
            raise ValueError("ring_index, producer_keys and blindings must have the same length")
        if any(not 0 <= k < len(rings) for k in index):
            raise ValueError("ring index out of range")
        if transcript_label is not None and len(transcript_label) > 32:
            raise ValueError("transcript label longer than 32 bytes")
        if n == 0:
            return []
        order = rings[0].params.cv.curve.params.subgroup_order
        ts = [int(t) for t in blindings]
        if any(not 0 <= t < order for t in ts):
            raise ValueError("blinding factor is not below the group order")
        rows = [rings[k].index_of(bytes(pk)) for k, pk in zip(index, producer_keys)]
        zk = _blinding_rows([rings[k] for k in index], zk_rows)
        natives = [r.native for r in rings]
        pooled = [isinstance(x, PooledRingNative) for x in natives]
        if any(pooled) and not all(pooled):
            raise ValueError("rings of one call must be built on the same engine")
        prove = PooledRingNative.proof_prove_multi if all(pooled) else _native.NativeRing.proof_prove_multi
        relations, payloads = prove(natives, index, rows, ts, zk, transcript_label)
        return [cls(r, p) for r, p in zip(relations, payloads)]

    @staticmethod
    def verify_batch(proofs, relations: Sequence[tuple[int, int]], ring_root: RingRoot, transcript_label: bytes | None = None, aggregate: bool = False):
        """`Verify(...).is_valid()` (ring_proof/verify.py:213-324) for (relation, proof) pairs against ``ring_root`` under
        ``transcript_label`` (default: the suite id).  The verifier key is the root's fixed commitments with [1]_1 and the G2 points of
        the root's engine.  Per item (default): one verdict per proof, 1 valid, 0 invalid, 2 malformed.  ``aggregate=True``: one
        pairing check over the whole batch -> bool."""
        from .kzg import _random_nonzero_coefficients

        if ring_root.params is None:
            raise ValueError("ring-proof verification requires the root's ring proof parameters")
        raw = [bytes(p) if isinstance(p, (bytes, bytearray)) else p.encode() for p in proofs]
        n = len(raw)
        if len(relations) != n:
            raise ValueError("proofs and relations must have the same length")
        if any(len(p) != RING_PAYLOAD_LEN for p in raw):
            raise ValueError(f"invalid ring proof length: ring proof must be exactly {RING_PAYLOAD_LEN} bytes")
        params = ring_root.params
        suite = params.cv.curve.params
        label = suite.suite_id if transcript_label is None else bytes(transcript_label)
        engine = ring_root.engine or default_engine()
        srs = engine.srs_bytes  # [1]_1 and the G2 points only: the window table is not built here
        key = _native.VerifierKeyStruct()
        key.domain_size = params.domain_size
        key.label_len = len(label)
        _native._put(key.label, label)
        _native._put(key.omega, int(params.omega).to_bytes(32, "little"))
        _native._put(key.seed, _native._xy64(suite.auxiliary_points.accumulator_base))
        _native._put(key.g1_0_be96, srs.g1_be96[:96])
        _native._put(key.g2_be192, srs.g2_be192)
        _native._put(key.fixed_be96, b"".join(ring_root.fixed_commitments()))
        if n == 0:
            return True if aggregate else []
        if aggregate:
            coeffs = _random_nonzero_coefficients(2 * n, params.prime)
        else:  # independent checks: (1, r) per proof
            coeffs = [v for r in _random_nonzero_coefficients(n + 1, params.prime)[1:] for v in (1, r)]
        ctx = engine.engines[0].ctx if isinstance(engine, EnginePool) else engine.ctx
        verdicts, all_ok = ctx.ring_proof_verify(key, [tuple(r) for r in relations], raw, coeffs, aggregate)
        return all_ok if aggregate else verdicts


__all__ = ["RingProof"]
