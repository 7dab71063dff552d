"""Bare ring proofs from a caller's blinding factor (dr_ring_proof_prove_multi, NativeRing.proof_prove_multi, RingProof): cases shared by
the CPU (emulation build) and GPU (CUDA build) suites.

A Ring VRF proof is its Pedersen part (which fixes the blinding factor t) followed by the ring proof of relation = PK_k + t * B.  So a
bare ring proof made with the t of `PedersenVRF.prove` must equal bytes 192..784 of the Ring VRF proof, and its relation the proof's
blinded key (bytes 32..64): that pins the bare prover to the reference's vectors.  Other labels are pinned by the CPU oracle."""

from __future__ import annotations

import random

from dot_ring_b200 import _native
from dot_ring_b200.srs import read_srs_file
from oracle import bandersnatch as bs
from oracle import fr
from oracle import ring_proof as rp
from tests import ring_prove_multi_cases as pm
from tests.helpers import hx, load, ring_proof_bytes, split_keys
from tests.ring_fixtures import native_ring
from tests.verify_cases import SUITES, coeffs_for, suite_struct

W3F = b"w3f-ring-proof-test"


def refused(fn) -> bool:
    try:
        fn()
    except ValueError:
        return True
    return False


def blinding_factors(ctx, suite, alphas, ads, sks) -> list[int]:
    """`PedersenVRF.prove(...)._blinding_factor` of every item (dr_pedersen_prove_batch_ex)."""
    return ctx.pedersen_prove_with_blinding(suite_struct(suite), list(alphas), list(ads), list(sks))[1]


def blinded_key(proof784: bytes) -> tuple[int, int]:
    return bs.dec_point(proof784[32:64])


def verifier_key(ring: _native.NativeRing, params: rp.Params, label: bytes | None = None) -> _native.VerifierKeyStruct:
    """The dr_verifier_key of a native ring under `label` (None: the suite id)."""
    srs = read_srs_file(None, None)
    label = params.suite.suite_id if label is None else label
    key = _native.VerifierKeyStruct()
    key.domain_size = params.domain_size
    key.label_len = len(label)
    _native._put(key.label, label)
    _native._put(key.omega, params.omega.to_bytes(32, "little"))
    _native._put(key.seed, _native._xy64(params.suite.accumulator_base))
    _native._put(key.g1_0_be96, srs.g1_be96[:96])
    _native._put(key.g2_be192, srs.g2_be192)
    _native._put(key.fixed_be96, ring.fixed_commitments())
    return key


def prove(natives, items, ts, label=None, zk=True):
    """NativeRing.proof_prove_multi of ring_prove_multi_cases items with blinding factors `ts` -> (relations, payloads)."""
    return _native.NativeRing.proof_prove_multi(natives, [it[0] for it in items], [it[5] for it in items], ts, pm.zk_of(items) if zk else None, label)


# ---- 1. composition with the Pedersen prover pins the bytes to the reference --------------------------------------------------------


def composition_ark_vectors(ctx, srs) -> None:
    """The seven ark-vrf ring vectors of both suites (ring 8, N = 512, zero rows), one call per suite over every ring of its vectors:
    with t from the Pedersen prover, the payload is bytes 192..784 of the vector's proof and the relation its blinded key."""
    for suite, name in SUITES:
        vecs = load(name + "_ring.json")
        assert len(vecs) == 7
        params = rp.Params(test_vectors=True, suite=suite)
        ring_keys = []
        for v in vecs:
            if hx(v, "ring_pks") not in ring_keys:
                ring_keys.append(hx(v, "ring_pks"))
        natives = [native_ring(srs, split_keys(k), params) for k in ring_keys]
        index = [ring_keys.index(hx(v, "ring_pks")) for v in vecs]
        rows = [split_keys(hx(v, "ring_pks")).index(hx(v, "pk")) for v in vecs]
        ts = blinding_factors(ctx, suite, [hx(v, "alpha") for v in vecs], [hx(v, "ad") for v in vecs], [hx(v, "sk") for v in vecs])
        relations, payloads = _native.NativeRing.proof_prove_multi(natives, index, rows, ts)
        for v, rel, pay in zip(vecs, relations, payloads):
            proof = ring_proof_bytes(v)
            assert pay == proof[192:], name
            assert rel == blinded_key(proof), name
        for r in natives:
            r.close()


def composition_ring1023(ctx, srs) -> None:
    """The reference-generated ring-1023 / N = 2048 proofs of ring1023_reference.json, with their zeroed and blinded rows."""
    rings, items = pm.reference_rings(with_2048=True)
    k = len(rings) - 1
    items = [it for it in items if it[0] == k]
    assert len(items) == 6
    native = native_ring(srs, *rings[k])
    ts = blinding_factors(ctx, bs.SHA512, [it[1] for it in items], [it[2] for it in items], [it[3] for it in items])
    relations, payloads = prove([native], [(0,) + it[1:] for it in items], ts)
    for it, rel, pay in zip(items, relations, payloads):
        assert pay == it[7][192:]
        assert rel == blinded_key(it[7])
    native.close()


# ---- 2. another transcript label, pinned by the oracle ------------------------------------------------------------------------------


def custom_label(ctx, srs, domain_size: int = 512) -> None:
    """Under "w3f-ring-proof-test", with zero rows and with given rows: byte-equal to oracle.ring_proof.prove_ring with that label.
    N = 512: the ark-vrf ring of eight keys; N = 2048: the ring of 1023 keys."""
    if domain_size == 512:
        v = load(SUITES[0][1] + "_ring.json")[0]
        keys, pk = split_keys(hx(v, "ring_pks")), hx(v, "pk")
        params = rp.Params()
    else:
        from tests.helpers import bench_ring_keys

        pk, _, keys = bench_ring_keys(1023)
        params = rp.Params.from_ring_size(1023)
    rng = random.Random(domain_size)
    native = native_ring(srs, keys, params)
    oring = rp.Ring(keys, params)
    oroot = rp.RingRoot.from_ring(oring, params)
    row = oring.index_of(pk)
    t = rng.randrange(bs.N)
    cases = [None, [rng.randrange(fr.R) for _ in range(12)]] if domain_size == 512 else [[rng.randrange(fr.R) for _ in range(12)]]
    for zk in cases:
        want = rp.prove_ring(oring, oroot, pk, t, zk_rows=zk or [0] * 12, transcript_label=W3F).encode()
        relations, payloads = _native.NativeRing.proof_prove_multi([native], [0], [row], [t], zk, W3F)
        assert payloads[0] == want, zk is None
        assert relations[0] == bs.add(oring.nm_points[row], bs.mul(params.suite.blinding_base, t))
        verdicts, _ = ctx.ring_proof_verify(verifier_key(native, params, W3F), relations, payloads, coeffs_for(1))
        assert verdicts == [1]
    native.close()


# ---- 3. round trip through the existing verifier ---------------------------------------------------------------------------------------


def round_trip(ctx, srs) -> None:
    """dr_ring_proof_verify_batch accepts every bare proof under its own label, per item and aggregated, and rejects it under the other
    label, against another ring's root, and with another item's relation."""
    rings, _ = pm.reference_rings()
    natives = pm.build(srs, rings)
    items = pm.shuffled_batch(rings, 1, 19)
    items = [it for it in items if it[0] in (0, 1)][:6]
    assert {it[0] for it in items} == {0, 1}
    rng = random.Random(3)
    ts = [rng.randrange(bs.N) for _ in items]
    for label, other in ((None, W3F), (W3F, None)):
        relations, payloads = prove(natives, items, ts, label)
        for k in (0, 1):
            sel = [i for i, it in enumerate(items) if it[0] == k]
            rel, pay = [relations[i] for i in sel], [payloads[i] for i in sel]
            n = len(sel)
            own, wrong_label = verifier_key(natives[k], rings[k][1], label), verifier_key(natives[k], rings[k][1], other)
            wrong_ring = verifier_key(natives[1 - k], rings[1 - k][1], label)
            assert ctx.ring_proof_verify(own, rel, pay, coeffs_for(n)) == ([1] * n, True)
            assert ctx.ring_proof_verify(own, rel, pay, coeffs_for(n, 5, independent=False), aggregate=True)[1]
            assert ctx.ring_proof_verify(wrong_label, rel, pay, coeffs_for(n))[0] == [0] * n
            assert not ctx.ring_proof_verify(wrong_label, rel, pay, coeffs_for(n, 5, independent=False), aggregate=True)[1]
            assert ctx.ring_proof_verify(wrong_ring, rel, pay, coeffs_for(n))[0] == [0] * n
            swapped = rel[1:] + rel[:1]
            assert ctx.ring_proof_verify(own, swapped, pay, coeffs_for(n))[0] == [0] * n
            assert not ctx.ring_proof_verify(own, swapped, pay, coeffs_for(n, 5, independent=False), aggregate=True)[1]
    for r in natives:
        r.close()


# ---- 4. several rings in one call -----------------------------------------------------------------------------------------------------


def several_rings(ctx, srs, with_2048: bool = False) -> None:
    """Interleaved items over the reference rings (N = 512 and, with `with_2048`, N = 2048): every proof equals the one-ring call on
    the same item; passes of two, the generic NTT path and the dense witness commit give the same bytes; with the Pedersen prover's t
    every payload is the tail of dr_ring_prove_multi's proof."""
    rings, _ = pm.reference_rings(with_2048)
    natives = pm.build(srs, rings)
    items = pm.shuffled_batch(rings, 2, 23, with_2048)
    rng = random.Random(29)
    ts = [rng.randrange(bs.N) for _ in items]
    want = prove(natives, items, ts)
    for k, ring in enumerate(natives):
        for i, it in enumerate(items):
            if it[0] == k:
                got = _native.NativeRing.proof_prove_multi([ring], [0], [it[5]], [ts[i]], it[6], None)
                assert (got[0][0], got[1][0]) == (want[0][i], want[1][i]), i
    for name, on, off in (
        ("passes of two", lambda: ctx.set_prove_chunk(2), lambda: ctx.set_prove_chunk(0)),
        ("generic NTT path", lambda: ctx.set_generic_ntt_path(True), lambda: ctx.set_generic_ntt_path(False)),
        ("dense witness commit", lambda: ctx.set_dense_witness_commit(True), lambda: ctx.set_dense_witness_commit(False)),
    ):
        on()
        try:
            assert prove(natives, items, ts) == want, name
        finally:
            off()
    # composition over several rings: t of the Pedersen prover -> the tail of the Ring VRF proofs
    ped = blinding_factors(ctx, bs.SHA512, [it[1] for it in items], [it[2] for it in items], [it[3] for it in items])
    proofs, status = pm.prove_multi(natives, items)
    assert status == [0] * len(items)
    relations, payloads = prove(natives, items, ped)
    assert payloads == [p[192:] for p in proofs]
    assert relations == [blinded_key(p) for p in proofs]
    for r in natives:
        r.close()


# ---- 5. arguments ------------------------------------------------------------------------------------------------------------------


def errors(ctx, srs, other_srs) -> None:
    """DR_EINVAL / ValueError for t >= order, a row >= max_ring_size, a 33-byte label, rings on different SRS handles and an index out
    of range; n == 0 proves nothing; a row holding the padding point is proved and verifies."""
    rings, items = pm.reference_rings()
    natives = pm.build(srs, rings)
    it = items[0]
    ok = lambda **kw: _native.NativeRing.proof_prove_multi(natives, [kw.get("k", 0)], [kw.get("row", it[5])], [kw.get("t", 5)], None, kw.get("label"))  # noqa: E731
    ok()
    ok(t=bs.N - 1)
    ok(label=b"x" * 32)
    assert refused(lambda: ok(t=bs.N))
    assert refused(lambda: ok(t=(1 << 256) - 1))
    assert refused(lambda: ok(row=rings[0][1].max_ring_size))
    assert refused(lambda: ok(label=b"x" * 33))
    assert refused(lambda: ok(k=len(natives)))
    twin = native_ring(other_srs, *rings[0])
    assert refused(lambda: _native.NativeRing.proof_prove_multi(natives + [twin], [0], [it[5]], [5]))
    twin.close()
    lib = ctx.library.lib
    assert lib.dr_ring_proof_prove_multi(ctx.handle, None, 0, None, 0, None, None, None, None, 0, None, None) == _native.DR_OK
    assert lib.dr_ring_proof_prove_multi(ctx.handle, None, 0, None, 0, None, None, None, b"x" * 33, 33, None, None) == _native.DR_EINVAL
    assert _native.NativeRing.proof_prove_multi(natives, [], [], []) == ([], [])
    # ring 0 holds eight keys below max_ring_size 255: row 100 is the padding point
    keys, params = rings[0]
    pad_row = 100
    assert len(keys) < pad_row < params.max_ring_size
    t = 12345
    relations, payloads = _native.NativeRing.proof_prove_multi(natives, [0], [pad_row], [t])
    assert relations[0] == bs.add(params.suite.padding_point, bs.mul(params.suite.blinding_base, t))
    assert ctx.ring_proof_verify(verifier_key(natives[0], params), relations, payloads, coeffs_for(1))[0] == [1]
    for r in natives:
        r.close()


# ---- API: RingProof ------------------------------------------------------------------------------------------------------------------


def api_round_trip(api, engine) -> None:
    """RingProof.prove_batch with PedersenVRF's blinding factors gives the tail of RingVRF.prove; RingProof.verify_batch accepts the
    proofs under their label, per item and aggregated, and rejects them under another label or another item's relation; a key that
    is not in the ring, a blinding factor out of range and a long label raise ValueError."""
    rings, items = pm.reference_rings()
    objs = pm.api_rings(api, engine, rings)
    ring, root = objs[0], api.RingRoot.from_ring(objs[0])
    sel = [x for x in items if x[0] == 0][:1] + [x for x in pm.extra_items(rings, items, 3, 31) if x[0] == 0]
    alphas, ads, sks, pks = [x[1] for x in sel], [x[2] for x in sel], [x[3] for x in sel], [x[4] for x in sel]
    ped = api.PedersenVRF[api.Bandersnatch].prove_batch(alphas, sks, ads)
    ts = [p._blinding_factor for p in ped]
    vrf = api.RingVRF[api.Bandersnatch].prove_batch(alphas, ads, sks, pks, ring, as_bytes=True)
    proofs = api.RingProof.prove_batch(ring, pks, ts)
    assert [p.encode() for p in proofs] == [v[192:] for v in vrf]
    assert [p.relation for p in proofs] == [blinded_key(v) for v in vrf]
    assert sel[0][7] is not None and proofs[0].payload == sel[0][7][192:]
    n = len(proofs)
    rel = [p.relation for p in proofs]
    assert api.RingProof.verify_batch(proofs, rel, root) == [1] * n
    assert api.RingProof.verify_batch(proofs, rel, root, aggregate=True)
    assert api.RingProof.verify_batch(proofs, rel, root, transcript_label=W3F) == [0] * n
    assert api.RingProof.verify_batch(proofs, rel[1:] + rel[:1], root) == [0] * n
    w3f = api.RingProof.prove_batch(ring, pks, ts, transcript_label=W3F)
    assert api.RingProof.verify_batch(w3f, rel, root, transcript_label=W3F) == [1] * n
    assert not api.RingProof.verify_batch(w3f, rel, root, aggregate=True)
    # a blinded ring (test_vectors=False) with given rows, through prove_multi, against the native call
    k = [i for i, r in enumerate(objs) if not r.params.test_vectors][0]
    zk = [random.Random(37).randrange(fr.R) for _ in range(12 * 2)]
    signer = [x for x in items if x[0] == k][0]
    multi = api.RingProof.prove_multi(objs, [k, 0], [signer[4], pks[0]], [7, 9], zk_rows=zk, transcript_label=W3F)
    assert multi[0].payload == _native.NativeRing.proof_prove_multi([objs[k].native], [0], [signer[5]], [7], zk[:12], W3F)[1][0]
    assert multi[1].payload == _native.NativeRing.proof_prove_multi([ring.native], [0], [sel[0][5]], [9], None, W3F)[1][0]
    assert api.RingProof.verify_batch(multi[:1], [multi[0].relation], api.RingRoot.from_ring(objs[k]), transcript_label=W3F) == [1]
    fresh = api.RingProof.prove_multi(objs, [k], [signer[4]], [7])  # fresh rows
    assert fresh[0].relation == multi[0].relation and fresh[0].payload != multi[0].payload
    outsider = api.Bandersnatch.public_keys_from_secrets([bytes.fromhex(load(SUITES[0][1] + "_ring.json")[1]["sk"])])[0]
    outside = [i for i, (keys, _) in enumerate(rings) if outsider not in keys][0]
    assert refused(lambda: api.RingProof.prove_batch(objs[outside], [outsider], [1]))
    assert refused(lambda: api.RingProof.prove_batch(ring, pks[:1], [bs.N]))
    assert refused(lambda: api.RingProof.prove_batch(ring, pks[:1], [1], transcript_label=b"x" * 33))
    assert refused(lambda: api.RingProof.prove_multi(objs, [len(objs)], pks[:1], [1]))
    assert api.RingProof.prove_batch(ring, [], []) == []


def pool_matches_one_engine(api, engine, pool, with_2048: bool = False) -> None:
    """RingProof.prove_multi over rings built on a two-device EnginePool gives the bytes of the same rings on one engine."""
    rings, _ = pm.reference_rings(with_2048)
    one = pm.api_rings(api, engine, rings)
    many = pm.api_rings(api, pool, rings)
    items = pm.shuffled_batch(rings, 2, 41, with_2048)
    rng = random.Random(43)
    ts = [rng.randrange(bs.N) for _ in items]
    args = ([it[0] for it in items], [it[4] for it in items], ts)
    zk = pm.zk_of(items)
    for label in (None, W3F):
        want = api.RingProof.prove_multi(one, *args, zk_rows=zk, transcript_label=label)
        assert api.RingProof.prove_multi(many, *args, zk_rows=zk, transcript_label=label) == want
    assert refused(lambda: api.RingProof.prove_multi([one[0]] + many[1:], *args, zk_rows=zk))
    for r in one + many:
        r.native.close()


# ---- 6. full size (GPU) ----------------------------------------------------------------------------------------------------------------


def full_size_4096(ctx, srs) -> None:
    """4096 bare proofs at ring 1023 over eight rings, with the Pedersen prover's blinding factors: a 64-proof sample equals the tail
    of dr_ring_prove_multi's Ring VRF proofs and their blinded keys."""
    keys, params, items = pm.eight_rings_1023(srs)
    assert len(items) == 4096
    natives = [native_ring(srs, k, params) for k in keys]
    ts = blinding_factors(ctx, bs.SHA512, [it[1] for it in items], [it[2] for it in items], [it[3] for it in items])
    relations, payloads = prove(natives, items, ts)
    sample = random.Random(47).sample(range(len(items)), 64)
    proofs, status = pm.prove_multi(natives, [items[i] for i in sample])
    assert status == [0] * 64
    for i, p in zip(sample, proofs):
        assert payloads[i] == p[192:], i
        assert relations[i] == blinded_key(p), i
    for r in natives:
        r.close()

