"""RingVRF / PedersenVRF: drop-in mirrors of dot_ring/vrf/ring/vrf.py:30-294 and
dot_ring/vrf/pedersen/vrf.py:33-242 for the Bandersnatch suite, with batched entry points.

``RingVRF[Bandersnatch].prove(alpha, ad, sk, pk, ring, ring_root)`` keeps the reference signature and
is ``prove_batch`` with one item; ``prove_batch`` is the call the 4096-proof configuration uses.
Blinding rows: ``RingProofParams(test_vectors=True)`` -> zeros (as in the reference);
otherwise 12 fresh ``secrets.randbelow(prime)`` values per proof in the reference's draw order
(b, acc_x, acc_y, acc_ip; columns.py:43-53,153-161) unless ``zk_rows`` injects them.
"""

from __future__ import annotations

import hashlib
import secrets
from collections.abc import Sequence
from dataclasses import dataclass
from typing import Any, ClassVar

from .curve import Bandersnatch, CurveVariant
from .ring import Column, Ring, RingRoot

PEDERSEN_LEN = 192
RING_PAYLOAD_LEN = 592
RING_PROOF_LEN = PEDERSEN_LEN + RING_PAYLOAD_LEN


class VRF:
    """vrf/vrf.py:12-28: ``Scheme[curve]`` specialisation by subscription."""

    cv: ClassVar[CurveVariant] = Bandersnatch

    def __class_getitem__(cls, curve_variant: Any):
        if not isinstance(curve_variant, CurveVariant):
            return cls
        return type(f"{cls.__name__}[{curve_variant.name}]", (cls,), {"cv": curve_variant})


def _dec_scalar(cv: CurveVariant, value: bytes) -> int:
    if len(value) != 32:
        raise ValueError("scalar must be exactly 32 bytes")
    scalar = int.from_bytes(value, "little")
    if scalar >= cv.curve.params.subgroup_order:
        raise ValueError("scalar is not canonical")
    return scalar


from .kzg import _random_nonzero_coefficients  # noqa: E402  (pcs/kzg.py:84-108)


def _suite_struct(cv: CurveVariant):
    from . import _native

    p = cv.curve.params
    return _native.make_suite(p.suite_id, p.hash_to_curve.dst, p.generator, p.auxiliary_points.blinding_base, p.hash_name)


def _point_to_hash(cv: CurveVariant, point: bytes, size: int = 32) -> bytes:
    """primitives.py:91-96 over the 32-byte encoding of the output point."""
    from .transcript import _squeeze

    return _squeeze(cv.curve.params.suite_id + bytes([0x20]) + bytes(point), size, cv.curve.params.hash_name)


@dataclass(frozen=True)
class TinyVRF(VRF):
    """ietf/tiny.py:27-89: gamma (32) | c (16) | s (32)."""

    output_point: bytes
    c: int
    s: int

    @classmethod
    def proof_len(cls) -> int:
        return 80

    @classmethod
    def decode(cls, proof: bytes) -> "TinyVRF":
        if len(proof) != 80:
            raise ValueError(f"invalid Tiny VRF proof length: expected 80, got {len(proof)}")
        from .engine import default_engine

        proof = bytes(proof)
        if default_engine().ctx.te_decode([proof[:32]], checked=True)[0] is None:
            raise ValueError("Invalid output point")
        return cls(proof[:32], int.from_bytes(proof[32:48], "little"), _dec_scalar(cls.cv, proof[48:80]))

    def encode(self) -> bytes:
        return self.output_point + self.c.to_bytes(16, "little") + self.s.to_bytes(32, "little")

    @classmethod
    def prove(cls, alpha: bytes, secret_key: bytes, additional_data: bytes, salt: bytes = b"") -> "TinyVRF":
        return cls.prove_batch([alpha], [secret_key], [additional_data], [salt])[0]

    @classmethod
    def prove_batch(cls, alphas, secret_keys, additional_data, salts=None, as_bytes: bool = False):
        from .engine import default_engine

        salts = salts or [b""] * len(alphas)
        raw = default_engine().ctx.vrf_prove(
            "tiny", _suite_struct(cls.cv), [bytes(s) + bytes(a) for s, a in zip(salts, alphas, strict=True)], [bytes(d) for d in additional_data], [bytes(k) for k in secret_keys]
        )
        if as_bytes:
            return raw
        return [cls(p[:32], int.from_bytes(p[32:48], "little"), int.from_bytes(p[48:], "little")) for p in raw]

    def verify(self, public_key: bytes, input: bytes, additional_data: bytes, salt: bytes = b"") -> bool:
        """ietf/tiny.py:72-83; an undecodable public key raises ValueError as in the reference."""
        verdict = self.verify_batch([self.encode()], [public_key], [input], [additional_data], [salt])[0]
        if verdict == 2:
            raise ValueError("Invalid public key")
        return verdict == 1

    @classmethod
    def verify_batch(cls, proofs, public_keys, inputs, additional_data, salts=None) -> list[int]:
        """Independent verifications (the reference has no batch equation for Tiny): 1 valid, 0 invalid, 2 malformed."""
        from .engine import default_engine

        salts = salts or [b""] * len(proofs)
        raw = [p if isinstance(p, (bytes, bytearray)) else p.encode() for p in proofs]
        return default_engine().ctx.tiny_verify(
            _suite_struct(cls.cv), [bytes(k) for k in public_keys], [bytes(s) + bytes(a) for s, a in zip(salts, inputs, strict=True)], [bytes(d) for d in additional_data], [bytes(p) for p in raw]
        )

    @classmethod
    def proof_to_hash(cls, gamma: bytes, mul_cofactor: bool = False) -> bytes:
        return PedersenVRF[cls.cv].proof_to_hash(gamma, mul_cofactor)


@dataclass(frozen=True)
class ThinVRF(VRF):
    """ietf/thin.py:38-152: gamma (32) | R (32) | s (32)."""

    output_point: bytes
    r: bytes
    s: int

    @classmethod
    def proof_len(cls) -> int:
        return 96

    @classmethod
    def decode(cls, proof: bytes) -> "ThinVRF":
        if len(proof) != 96:
            raise ValueError(f"invalid Thin VRF proof length: expected 96, got {len(proof)}")
        from .engine import default_engine

        proof = bytes(proof)
        if any(p is None for p in default_engine().ctx.te_decode([proof[:32], proof[32:64]], checked=True)):
            raise ValueError("Invalid point encoding")
        return cls(proof[:32], proof[32:64], _dec_scalar(cls.cv, proof[64:96]))

    def encode(self) -> bytes:
        return self.output_point + self.r + self.s.to_bytes(32, "little")

    @classmethod
    def prove(cls, alpha: bytes, secret_key: bytes, additional_data: bytes, salt: bytes = b"") -> "ThinVRF":
        return cls.prove_batch([alpha], [secret_key], [additional_data], [salt])[0]

    @classmethod
    def prove_batch(cls, alphas, secret_keys, additional_data, salts=None, as_bytes: bool = False):
        from .engine import default_engine

        salts = salts or [b""] * len(alphas)
        raw = default_engine().ctx.vrf_prove(
            "thin", _suite_struct(cls.cv), [bytes(s) + bytes(a) for s, a in zip(salts, alphas, strict=True)], [bytes(d) for d in additional_data], [bytes(k) for k in secret_keys]
        )
        if as_bytes:
            return raw
        return [cls(p[:32], p[32:64], int.from_bytes(p[64:], "little")) for p in raw]

    def verify(self, public_key: bytes, input: bytes, additional_data: bytes, salt: bytes = b"") -> bool:
        """ietf/thin.py:84-99; an undecodable public key raises ValueError as in the reference."""
        if len(public_key) != 32:
            raise ValueError("Invalid public key")
        from .engine import default_engine

        if default_engine().ctx.te_decode([bytes(public_key)], checked=True)[0] is None:
            raise ValueError("Invalid public key")
        return self.verify_batch([self], [public_key], [input], [additional_data], [salt])[0] == 1

    @classmethod
    def verify_batch(cls, proofs, public_keys, inputs, additional_data, salts=None) -> list[int]:
        """Per-item verdicts: 1 valid, 0 invalid, 2 malformed."""
        from .engine import default_engine

        salts = salts or [b""] * len(proofs)
        raw = [bytes(p) if isinstance(p, (bytes, bytearray)) else p.encode() for p in proofs]
        return default_engine().ctx.thin_verify(
            _suite_struct(cls.cv), [bytes(k) for k in public_keys], [bytes(s) + bytes(a) for s, a in zip(salts, inputs, strict=True)], [bytes(d) for d in additional_data], raw
        )

    @classmethod
    def batch_verify(cls, proofs, public_keys, inputs, additional_data, salts=None) -> bool:
        """ietf/thin.py:108-152: True iff every proof verifies; malformed input / mismatched lengths -> False."""
        try:
            if not (len(proofs) == len(public_keys) == len(inputs) == len(additional_data)) or (salts is not None and len(salts) != len(proofs)):
                return False
            return all(v == 1 for v in cls.verify_batch(proofs, public_keys, inputs, additional_data, salts))
        except (AssertionError, AttributeError, TypeError, ValueError):
            return False

    @classmethod
    def proof_to_hash(cls, gamma: bytes, mul_cofactor: bool = False) -> bytes:
        return PedersenVRF[cls.cv].proof_to_hash(gamma, mul_cofactor)


@dataclass(frozen=True)
class PedersenVRF(VRF):
    """gamma || Y_bar || R || O_k || s || s_b (points as 32-byte encodings)."""

    output_point: bytes
    blinded_pk: bytes
    result_point: bytes
    ok: bytes
    s: int
    sb: int
    _blinding_factor: int | None = None  # known to the prover only (pedersen/vrf.py:44, 111-126)

    @classmethod
    def proof_len(cls) -> int:
        return PEDERSEN_LEN

    @classmethod
    def decode(cls, proof: bytes) -> "PedersenVRF":
        """pedersen/vrf.py:48-73: four validated subgroup points and two canonical scalars."""
        if len(proof) != PEDERSEN_LEN:
            raise ValueError(f"invalid Pedersen VRF proof length: expected {PEDERSEN_LEN}, got {len(proof)}")
        from .engine import default_engine

        pts = [bytes(proof[32 * i : 32 * i + 32]) for i in range(4)]
        if any(p is None for p in default_engine().ctx.te_decode(pts, checked=True)):
            raise ValueError("Invalid point in proof")
        return cls(pts[0], pts[1], pts[2], pts[3], _dec_scalar(cls.cv, proof[128:160]), _dec_scalar(cls.cv, proof[160:192]))

    def encode(self) -> bytes:
        return self.output_point + self.blinded_pk + self.result_point + self.ok + self.s.to_bytes(32, "little") + self.sb.to_bytes(32, "little")

    @classmethod
    def prove(cls, alpha: bytes, secret_key: bytes, additional_data: bytes, salt: bytes = b"") -> "PedersenVRF":
        """pedersen/vrf.py:86-126."""
        return cls.prove_batch([alpha], [secret_key], [additional_data], [salt])[0]

    @classmethod
    def prove_batch(cls, alphas, secret_keys, additional_data, salts=None, as_bytes: bool = False):
        from .engine import default_engine

        salts = salts or [b""] * len(alphas)
        raw, blind = default_engine().ctx.pedersen_prove_with_blinding(
            _suite_struct(cls.cv), [bytes(s) + bytes(a) for s, a in zip(salts, alphas, strict=True)], [bytes(d) for d in additional_data], [bytes(k) for k in secret_keys]
        )
        if as_bytes:
            return raw
        return [
            cls(p[0:32], p[32:64], p[64:96], p[96:128], int.from_bytes(p[128:160], "little"), int.from_bytes(p[160:192], "little"), b)
            for p, b in zip(raw, blind)
        ]

    def verify_unblinding(self, public_key: bytes, blinding_factor: int) -> bool:
        """pedersen/vrf.py:144-156: Y_bar == Y + b * B for a revealed blinding factor."""
        from .engine import default_engine

        params = self.cv.curve.params
        if not 0 <= blinding_factor < params.subgroup_order:
            return False
        ctx = default_engine().ctx
        if len(public_key) != 32 or ctx.te_decode([bytes(public_key)], checked=True)[0] is None:
            raise ValueError("Invalid point encoding")
        from .curve import point_to_string

        return ctx.te_msm([bytes(public_key), point_to_string(params.auxiliary_points.blinding_base)], [1, blinding_factor]) == self.blinded_pk

    def verify(self, input: bytes, additional_data: bytes, salt: bytes = b"") -> bool:
        """pedersen/vrf.py:128-143."""
        return self.verify_batch([self], [input], [additional_data], [salt])[0] == 1

    @classmethod
    def verify_batch(cls, proofs, inputs, additional_data, salts=None) -> list[int]:
        """Per-item verdicts for a batch: 1 valid, 0 invalid, 2 malformed."""
        from .engine import default_engine

        salts = salts or [b""] * len(proofs)
        raw = [bytes(p) if isinstance(p, (bytes, bytearray)) else p.encode() for p in proofs]
        return default_engine().ctx.pedersen_verify(
            _suite_struct(cls.cv), [bytes(s) + bytes(a) for s, a in zip(salts, inputs, strict=True)], [bytes(d) for d in additional_data], raw
        )

    @classmethod
    def batch_verify(cls, proofs, inputs, additional_data, salts=None) -> bool:
        """pedersen/vrf.py:171-242: True iff every proof verifies (mismatched lengths / malformed input -> False)."""
        try:
            if not (len(proofs) == len(inputs) == len(additional_data)) or (salts is not None and len(salts) != len(proofs)):
                return False
            return all(v == 1 for v in cls.verify_batch(proofs, inputs, additional_data, salts))
        except (AssertionError, AttributeError, TypeError, ValueError):
            return False

    @classmethod
    def proof_to_hash(cls, gamma: bytes, mul_cofactor: bool = False) -> bytes:
        """pedersen/vrf.py:165-168 on the 32-byte encoding of gamma."""
        if mul_cofactor:
            from .engine import default_engine

            gamma = default_engine().ctx.te_mul([bytes(gamma)], [cls.cv.curve.params.cofactor])[0]
            if gamma is None:
                raise ValueError("Invalid point")
        return _point_to_hash(cls.cv, gamma)


@dataclass
class RingVRF(VRF):
    pedersen_proof: PedersenVRF
    c_b: Column
    c_accip: Column
    c_accx: Column
    c_accy: Column
    px_zeta: int
    py_zeta: int
    s_zeta: int
    b_zeta: int
    accip_zeta: int
    accx_zeta: int
    accy_zeta: int
    c_q: Column
    l_zeta_omega: int
    open_agg_zeta: bytes
    open_l_zeta_omega: bytes
    _encoded: bytes | None = None

    @classmethod
    def proof_len(cls) -> int:
        return RING_PROOF_LEN

    def encode(self) -> bytes:
        """vrf/ring/vrf.py:56-58 + proof_payload.py:68-91."""
        if self._encoded is not None:
            return self._encoded
        from .kzg import KZG

        le = lambda v: int(v).to_bytes(32, "little")  # noqa: E731
        g = KZG.compress_g1(
            self.c_b.commitment + self.c_accip.commitment + self.c_accx.commitment + self.c_accy.commitment + self.c_q.commitment
            + self.open_agg_zeta + self.open_l_zeta_omega
        )
        return (
            self.pedersen_proof.encode() + g[0:192]
            + b"".join(le(v) for v in (self.px_zeta, self.py_zeta, self.s_zeta, self.b_zeta, self.accip_zeta, self.accx_zeta, self.accy_zeta))
            + g[192:240] + le(self.l_zeta_omega) + g[240:288] + g[288:336]
        )  # fmt: skip

    @classmethod
    def decode(cls, proof: bytes) -> "RingVRF":
        """vrf/ring/vrf.py:60-93 + proof_payload.py:93-143: lengths, G1 / point validity, canonical scalars."""
        if len(proof) != RING_PROOF_LEN:
            raise ValueError(f"invalid Ring VRF proof length: Ring VRF proof must be exactly {RING_PROOF_LEN} bytes, got {len(proof)}")
        from .kzg import KZG

        proof = bytes(proof)
        pedersen = PedersenVRF[cls.cv].decode(proof[:PEDERSEN_LEN])
        body = proof[PEDERSEN_LEN:]
        prime = cls.cv.curve.params.field_modulus
        g1 = KZG.decompress_g1_batch(body[0:192] + body[416:464] + body[496:592])
        scalars = [int.from_bytes(body[192 + 32 * i : 224 + 32 * i], "little") for i in range(7)] + [int.from_bytes(body[464:496], "little")]
        if any(v >= prime for v in scalars):
            raise ValueError("scalar is not canonical")
        return cls(
            pedersen,
            Column("c_b", g1[0]), Column("c_accip", g1[1]), Column("c_accx", g1[2]), Column("c_accy", g1[3]),
            *scalars[:7],
            Column("c_q", g1[4]), scalars[7], g1[5], g1[6], _encoded=proof,
        )  # fmt: skip

    @classmethod
    def _from_bytes_trusted(cls, proof: bytes) -> "RingVRF":
        """Wrap device output without re-validating (points were produced by the prover itself)."""
        return _LazyRingVRF.wrap(cls, proof)

    @classmethod
    def parse_keys(cls, keys: bytes) -> list[bytes]:
        if len(keys) % 32 != 0:
            raise ValueError(f"invalid concatenated key length: expected multiple of 32, got {len(keys)}")
        return [keys[32 * i : 32 * (i + 1)] for i in range(len(keys) // 32)]

    # ---- proving -----------------------------------------------------------------------------
    @classmethod
    def prove(
        cls,
        alpha: bytes,
        additional_data: bytes,
        secret_key: bytes,
        producer_key: bytes,
        ring: Ring,
        ring_root: RingRoot | None = None,
        salt: bytes = b"",
        zk_rows: Sequence[int] | None = None,
    ) -> "RingVRF":
        """vrf/ring/vrf.py:185-209."""
        return cls.prove_batch([alpha], [additional_data], secret_key, producer_key, ring, ring_root, salt=salt, zk_rows=zk_rows)[0]

    @classmethod
    def _signer_rows(cls, ring: Ring, pairs) -> dict[bytes, int]:
        """{producer key: its row in `ring`} for a set of (secret key, producer key) pairs.  vrf.py:196-197: producer_key must be
        pk(sk) -- one device scalar multiplication per distinct key pair, remembered per ring under a digest of the pair (no secret
        key outlives the call in the cache); ValueError on a pair that does not match or a key that is not in the ring."""
        cache = ring.__dict__.setdefault("_signer_rows", {})
        tag = lambda sk, pk: hashlib.blake2b(sk + pk, digest_size=16).digest()  # noqa: E731
        distinct = sorted(p for p in pairs if tag(*p) not in cache)
        if distinct:
            derived = cls.cv.public_keys_from_secrets([sk for sk, _ in distinct])
            for (sk, pk), got in zip(distinct, derived):
                if pk != got:
                    raise ValueError("producer_key does not match secret_key")
                cache[tag(sk, pk)] = ring.index_of(pk)
        return {pk: cache[tag(sk, pk)] for sk, pk in pairs}

    @classmethod
    def prove_batch(
        cls,
        alphas: Sequence[bytes],
        additional_data: Sequence[bytes],
        secret_key: bytes | Sequence[bytes],
        producer_key: bytes | Sequence[bytes],
        ring: Ring,
        ring_root: RingRoot | None = None,
        salt: bytes = b"",
        zk_rows: Sequence[int] | bytes | None = None,
        as_bytes: bool = False,
    ):
        """Prove ``len(alphas)`` items against one ring in one device pass; semantically a loop over ``prove``."""
        n = len(alphas)
        if len(additional_data) != n:
            raise ValueError("alphas and additional_data must have the same length")
        sks = [bytes(secret_key)] * n if isinstance(secret_key, (bytes, bytearray)) else [bytes(s) for s in secret_key]
        pks = [bytes(producer_key)] * n if isinstance(producer_key, (bytes, bytearray)) else [bytes(p) for p in producer_key]
        if len(sks) != n or len(pks) != n:
            raise ValueError("secret_key / producer_key must be single values or one per item")
        index = cls._signer_rows(ring, set(zip(sks, pks)))
        if ring_root is not None and ring_root.encode() != RingRoot.from_ring(ring).encode():
            raise ValueError("ring_root does not match ring")
        if zk_rows is None and not ring.params.test_vectors:
            prime = ring.params.prime
            zk_rows = [secrets.randbelow(prime) for _ in range(12 * n)]
        elif ring.params.test_vectors:
            zk_rows = None
        msgs = [bytes(salt) + bytes(a) for a in alphas]
        proofs, status = ring.native.prove_batch(msgs, [bytes(a) for a in additional_data], sks, [index[pk] for pk in pks], zk_rows)
        if any(status):
            raise ValueError("producer_key does not match secret_key")
        if as_bytes:
            return proofs
        return [cls._from_bytes_trusted(p) for p in proofs]

    @classmethod
    def prove_multi(
        cls,
        alphas: Sequence[bytes],
        additional_data: Sequence[bytes],
        secret_keys: Sequence[bytes],
        producer_keys: Sequence[bytes],
        rings: Sequence[Ring],
        ring_index: Sequence[int],
        salt: bytes = b"",
        zk_rows: Sequence[int] | bytes | None = None,
        as_bytes: bool = False,
    ):
        """Prove item i against ``rings[ring_index[i]]``, every ring in one device pass; semantically a loop over ``prove``.

        The rings share the suite and the engine (one :class:`Engine`, or one :class:`EnginePool` whose devices each take a
        contiguous shard); their domain sizes may differ.  Blinding rows as in ``prove_batch``: 12 per item, drawn fresh unless
        ``zk_rows`` gives them, and zeros for items whose ring has ``test_vectors=True``."""
        from . import _native
        from .engine import PooledRingNative

        n = len(alphas)
        rings = list(rings)
        index = [int(k) for k in ring_index]
        sks, pks = [bytes(s) for s in secret_keys], [bytes(p) for p in producer_keys]
        if not (len(additional_data) == len(sks) == len(pks) == len(index) == n):
            raise ValueError("alphas, additional_data, secret_keys, producer_keys and ring_index must have the same length")
        if any(not 0 <= k < len(rings) for k in index):
            raise ValueError("ring index out of range")
        if n == 0:
            return []
        rows = [0] * n
        for k in sorted(set(index)):
            items = [i for i in range(n) if index[i] == k]
            found = cls._signer_rows(rings[k], {(sks[i], pks[i]) for i in items})
            for i in items:
                rows[i] = found[pks[i]]
        zk = _blinding_rows([rings[k] for k in index], zk_rows)
        natives = [r.native for r in rings]
        pooled = [isinstance(x, PooledRingNative) for x in natives]
        if any(pooled) and not all(pooled):
            raise ValueError("rings of one call must be built on the same engine")
        prove = PooledRingNative.prove_multi if all(pooled) else _native.NativeRing.prove_multi
        msgs = [bytes(salt) + bytes(a) for a in alphas]
        proofs, status = prove(natives, index, msgs, [bytes(a) for a in additional_data], sks, rows, zk)
        if any(status):
            raise ValueError("producer_key does not match secret_key")
        if as_bytes:
            return proofs
        return [cls._from_bytes_trusted(p) for p in proofs]

    # ---- verification ------------------------------------------------------------------------
    @classmethod
    def _verify_common(cls, proofs, inputs, additional_data, ring: Ring, ring_root: RingRoot, aggregate: bool):
        """-> (per-item verdicts, all_ok).  vrf/ring/vrf.py:173-182 (`matches_ring`), 226-283."""
        raw = [bytes(p) if isinstance(p, (bytes, bytearray)) else p.encode() for p in proofs]
        n = len(raw)
        if not (len(inputs) == len(additional_data) == n):
            raise ValueError("proofs, inputs and additional_data must have the same length")
        if not ring_root.matches_ring(ring):
            return [0] * n, False
        if n == 0:
            return [], True
        order = ring.params.prime
        if aggregate:
            coeffs = _random_nonzero_coefficients(2 * n, order)
        else:  # independent checks: (1, r) per proof, as KZG.batch_verify draws for a single proof's two openings
            coeffs = [v for r in _random_nonzero_coefficients(n + 1, order)[1:] for v in (1, r)]
        return ring.native.verify_batch([bytes(a) for a in inputs], [bytes(d) for d in additional_data], raw, coeffs, aggregate)

    def verify(self, input: bytes, ad_data: bytes, ring: Ring, ring_root: RingRoot) -> bool:
        """vrf/ring/vrf.py:226-232."""
        return self._verify_common([self], [input], [ad_data], ring, ring_root, False)[0][0] == 1

    @classmethod
    def verify_batch(cls, proofs, inputs, additional_data, ring: Ring, ring_root: RingRoot) -> list[int]:
        """Independent verifications, one verdict per item: 1 valid, 0 invalid, 2 malformed encoding."""
        return cls._verify_common(proofs, inputs, additional_data, ring, ring_root, False)[0]

    @classmethod
    def batch_verify(cls, proofs, inputs, additional_data, ring: Ring, ring_root: RingRoot) -> bool:
        """vrf/ring/vrf.py:239-283: one aggregated pairing check for the whole batch; any error -> False."""
        try:
            return cls._verify_common(proofs, inputs, additional_data, ring, ring_root, True)[1]
        except (AssertionError, AttributeError, TypeError, ValueError):
            return False

    @classmethod
    def proof_to_hash(cls, gamma: bytes, mul_cofactor: bool = False) -> bytes:
        return PedersenVRF[cls.cv].proof_to_hash(gamma, mul_cofactor)


def _blinding_rows(item_rings: Sequence[Ring], zk_rows):
    """The 12 blinding rows of every item, for the item's ring: zeros where the ring has ``test_vectors=True``, else the given
    ``zk_rows`` (ints, or 32-byte little-endian values) or fresh ``secrets.randbelow`` draws; None when every item is zeroed."""
    n = len(item_rings)
    zeroed = [r.params.test_vectors for r in item_rings]
    if all(zeroed):
        return None
    if zk_rows is None:
        prime = item_rings[zeroed.index(False)].params.prime
        return [0 if z else secrets.randbelow(prime) for z in zeroed for _ in range(12)]
    if isinstance(zk_rows, (bytes, bytearray)):
        if len(zk_rows) != 12 * 32 * n:
            raise ValueError("zk_rows must hold 12 field elements per proof")
        zk_rows = [int.from_bytes(zk_rows[32 * j : 32 * j + 32], "little") for j in range(12 * n)]
    if len(zk_rows) != 12 * n:
        raise ValueError("zk_rows must hold 12 field elements per proof")
    return [0 if zeroed[j // 12] else int(v) for j, v in enumerate(zk_rows)]


class _LazyRingVRF:
    """Field access on prover output decodes on demand; ``encode()`` is free."""

    @staticmethod
    def wrap(cls, proof: bytes) -> "RingVRF":
        obj = object.__new__(cls)
        object.__setattr__(obj, "_encoded", proof)
        object.__setattr__(obj, "_lazy", True)
        return obj


def _lazy_getattr(self, name):
    if name.startswith("__") or not object.__getattribute__(self, "__dict__").get("_lazy"):
        raise AttributeError(name)
    full = type(self).decode(object.__getattribute__(self, "_encoded"))
    self.__dict__.update(full.__dict__)
    self.__dict__["_lazy"] = False
    return self.__dict__[name]


RingVRF.__getattr__ = _lazy_getattr  # type: ignore[attr-defined]
