"""Ring VRF proving over several rings in one call (dr_ring_prove_multi, NativeRing.prove_multi, RingVRF.prove_multi): cases shared by
the CPU (emulation build) and GPU (CUDA build) suites.

Every proof is pinned by dr_ring_prove_batch of its own ring on the same item and, where the unmodified reference produced it
(small_ring_reference.json, ring1023_reference.json, the ark-vrf ring vectors), by the reference's bytes."""

from __future__ import annotations

import random

from dot_ring_b200 import _native
from oracle import fr
from oracle import ring_proof as rp
from tests.helpers import hx, le64, load, ring_proof_bytes, split_keys
from tests.ring_fixtures import native_ring
from tests.verify_cases import SUITES

ZERO_ROWS = [0] * 12


def reference_rings(with_2048: bool = False):
    """(rings, items) with rings = [(keys, rp.Params)] and items = [(ring, alpha, ad, sk, pk, row, zk rows or None, reference proof)]:
    the first ark-vrf SHA-512 ring vector (N = 512), the small_ring_reference.json rings of max_ring_size 100 and 1 (N = 512) and, with
    `with_2048`, its max_ring_size 6 ring and the ring of 1023 keys of ring1023_reference.json (both N = 2048)."""
    rings, items = [], []
    v = load(SUITES[0][1] + "_ring.json")[0]
    keys = split_keys(hx(v, "ring_pks"))
    rings.append((keys, rp.Params(test_vectors=True)))
    items.append((0, hx(v, "alpha"), hx(v, "ad"), hx(v, "sk"), hx(v, "pk"), keys.index(hx(v, "pk")), None, ring_proof_bytes(v)))
    slot = {}
    for e in load("small_ring_reference.json"):
        if e["domain_size"] != 512 and not with_2048:
            continue
        shape = (e["domain_size"], e["max_ring_size"])
        keys = [bytes.fromhex(k) for k in e["keys"]]
        if shape not in slot:
            slot[shape] = len(rings)
            rings.append((keys, rp.Params(domain_size=shape[0], max_ring_size=shape[1], test_vectors=True)))
        pk = bytes.fromhex(e["pk"])
        zk = [int(z, 16) for z in e["zk_rows"]] or None
        items.append((slot[shape], bytes.fromhex(e["alpha"]), bytes.fromhex(e["ad"]), bytes.fromhex(e["sk"]), pk, keys.index(pk), zk, bytes.fromhex(e["proof"])))
    if with_2048:
        from tests.helpers import bench_ring_keys

        ref = load("ring1023_reference.json")
        pk, sk, keys = bench_ring_keys(1023)
        assert pk.hex() == ref["signer_pk"] and sk.hex() == ref["signer_sk"]
        params = rp.Params.from_ring_size(1023)
        rings.append((keys, params))
        for e in ref["proofs_test_vectors"] + ref["proofs_blinded"]:
            zk = [int(z, 16) for z in e.get("zk_rows", [])] or None
            items.append((len(rings) - 1, bytes.fromhex(e["alpha"]), bytes.fromhex(e["ad"]), sk, pk, ref["signer_index"], zk, bytes.fromhex(e["proof"])))
    return rings, items


def extra_items(rings, items, per_ring: int, seed: int):
    """`per_ring` more items on every ring (the signer of its reference item, new inputs, seeded blinding rows)."""
    rng = random.Random(seed)
    signer = {}
    for it in items:
        signer.setdefault(it[0], it[3:6])
    out = []
    for k in range(len(rings)):
        sk, pk, row = signer[k]
        for j in range(per_ring):
            out.append((k, b"multi-%d-" % k + le64(j), b"multi-ad-" + le64(j), sk, pk, row, [rng.randrange(fr.R) for _ in range(12)], None))
    return out


def zk_of(items) -> list[int]:
    return [v for it in items for v in (it[6] or ZERO_ROWS)]


def prove_multi(natives, items, zk=True):
    """NativeRing.prove_multi of a batch of items -> (proofs, status)."""
    return _native.NativeRing.prove_multi(
        natives, [it[0] for it in items], [it[1] for it in items], [it[2] for it in items], [it[3] for it in items], [it[5] for it in items],
        zk_of(items) if zk else None,
    )  # fmt: skip


def one_ring_at_a_time(natives, items) -> list[bytes]:
    """Each item's proof from dr_ring_prove_batch of its own ring (one call per ring, the ring's items in batch order)."""
    out = [None] * len(items)
    for k, ring in enumerate(natives):
        sel = [i for i, it in enumerate(items) if it[0] == k]
        if not sel:
            continue
        part = [items[i] for i in sel]
        proofs, status = ring.prove_batch([it[1] for it in part], [it[2] for it in part], [it[3] for it in part], [it[5] for it in part], zk_of(part))
        assert not any(status)
        for i, p in zip(sel, proofs):
            out[i] = p
    return out


def build(srs, rings):
    return [native_ring(srs, keys, params) for keys, params in rings]


def shuffled_batch(rings, per_ring: int, seed: int, with_2048: bool = False):
    _, items = reference_rings(with_2048)
    items = items + extra_items(rings, items, per_ring, seed)
    random.Random(seed).shuffle(items)
    return items


# ---- 1. / 2. same bytes as one ring at a time, on every route ---------------------------------------------------------------------


def same_bytes(ctx, srs, per_ring: int = 1, with_2048: bool = False) -> None:
    """Shuffled ring indices over the reference rings: every proof equals dr_ring_prove_batch of its ring and, for the reference's items,
    the reference's bytes; the dense witness commit, the two-pass NTT route and passes of two proofs give the same bytes."""
    rings, _ = reference_rings(with_2048)
    natives = build(srs, rings)
    items = shuffled_batch(rings, per_ring, 7, with_2048)
    assert len({it[0] for it in items}) == len(rings) >= 3
    want = one_ring_at_a_time(natives, items)
    for it, w in zip(items, want):
        if it[7] is not None:
            assert w == it[7]
    proofs, status = prove_multi(natives, items)
    assert status == [0] * len(items)
    assert proofs == want
    # the reference's test-vector items alone, blinding rows NULL (zeros)
    tv = [it for it in items if it[7] is not None and it[6] is None]
    assert prove_multi(natives, tv, zk=False) == ([it[7] for it in tv], [0] * len(tv))
    for name, on, off in (
        ("dense witness commit", lambda: ctx.set_dense_witness_commit(True), lambda: ctx.set_dense_witness_commit(False)),
        ("generic NTT path", lambda: ctx.set_generic_ntt_path(True), lambda: ctx.set_generic_ntt_path(False)),
        ("passes of two", lambda: ctx.set_prove_chunk(2), lambda: ctx.set_prove_chunk(0)),
    ):
        on()
        try:
            assert prove_multi(natives, items) == (want, [0] * len(items)), name
        finally:
            off()
    for r in natives:
        r.close()


# ---- 3. status per item ---------------------------------------------------------------------------------------------------------


def status_per_item(ctx, srs) -> None:
    """An item whose producer_index points at a row of its ring that holds another key gets a non-zero status; the other items of the
    batch are unaffected."""
    rings, _ = reference_rings()
    natives = build(srs, rings)
    items = shuffled_batch(rings, 1, 11)
    want = one_ring_at_a_time(natives, items)
    bad = [i for i, it in enumerate(items) if it[0] == 0][0]  # the ark-vrf ring has eight keys
    k, alpha, ad, sk, pk, row, zk, ref = items[bad]
    items[bad] = (k, alpha, ad, sk, pk, (row + 1) % len(rings[0][0]), zk, ref)
    proofs, status = prove_multi(natives, items)
    assert status[bad] != 0
    assert [s for i, s in enumerate(status) if i != bad] == [0] * (len(items) - 1)
    assert [p for i, p in enumerate(proofs) if i != bad] == [w for i, w in enumerate(want) if i != bad]
    for r in natives:
        r.close()


# ---- API: RingVRF.prove_multi, round trip through RingVerifier, key errors --------------------------------------------------------


def api_rings(api, engine, rings):
    """dot_ring_b200.Ring objects for the fixtures' rings (the max_ring_size 100 ring blinded, the others test vectors)."""
    out = []
    for keys, p in rings:
        tv = not (p.domain_size == 512 and p.max_ring_size == 100)
        params = api.RingProofParams(domain_size=p.domain_size, max_ring_size=p.max_ring_size, test_vectors=tv)
        out.append(api.Ring(keys, params, engine))
    return out


def api_round_trip(api, engine) -> None:
    """RingVRF.prove_multi gives the bytes of RingVRF.prove per item (zeros for test-vector rings, the given rows otherwise); every
    proof verifies through RingVerifier with its own ring index, per item and aggregated, and gets verdict 0 on another ring; a
    producer key that does not match its secret key or is not in its ring raises ValueError."""
    cls = api.RingVRF[api.Bandersnatch]
    rings, _ = reference_rings()
    objs = api_rings(api, engine, rings)
    items = shuffled_batch(rings, 1, 13)
    n = len(items)
    index = [it[0] for it in items]
    alphas, ads, sks, pks = [it[1] for it in items], [it[2] for it in items], [it[3] for it in items], [it[4] for it in items]
    zk = zk_of(items)
    proofs = cls.prove_multi(alphas, ads, sks, pks, objs, index, zk_rows=zk, as_bytes=True)
    for i, it in enumerate(items):
        ring = objs[it[0]]
        rows = None if ring.params.test_vectors else zk[12 * i : 12 * i + 12]
        assert proofs[i] == cls.prove(it[1], it[2], it[3], it[4], ring, zk_rows=rows).encode(), i
        if it[7] is not None and (it[6] is None) == ring.params.test_vectors:
            assert proofs[i] == it[7], i
    objects = cls.prove_multi(alphas, ads, sks, pks, objs, index)  # fresh blinding rows
    assert len(objects) == n and all(len(p.encode()) == 784 for p in objects)
    verifier = api.RingVerifier([api.RingRoot.from_ring(r) for r in objs], engine)
    rotated = [(k + 1) % len(objs) for k in index]
    for batch in (proofs, objects):
        assert verifier.verify_batch(batch, alphas, ads, index) == [1] * n
        assert verifier.batch_verify(batch, alphas, ads, index)
        assert verifier.verify_batch(batch, alphas, ads, rotated) == [0] * n
        assert not verifier.batch_verify(batch, alphas, ads, rotated)
    verifier.close()
    # salt is prepended to every input, as in prove_batch
    salted = cls.prove_multi(alphas[:2], ads[:2], sks[:2], pks[:2], objs, index[:2], salt=b"salt", zk_rows=zk[:24], as_bytes=True)
    assert salted == cls.prove_multi([b"salt" + a for a in alphas[:2]], ads[:2], sks[:2], pks[:2], objs, index[:2], zk_rows=zk[:24], as_bytes=True)

    def refused(fn) -> bool:
        try:
            fn()
        except ValueError:
            return True
        return False

    other_sk = bytes.fromhex(load(SUITES[0][1] + "_ring.json")[1]["sk"])
    assert refused(lambda: cls.prove_multi(alphas, ads, [other_sk] + sks[1:], pks, objs, index))  # sk does not give pk
    outsider = api.Bandersnatch.public_keys_from_secrets([other_sk])[0]
    ring1 = [k for k, (keys, _) in enumerate(rings) if outsider not in keys][0]
    assert refused(lambda: cls.prove_multi(alphas[:1], ads[:1], [other_sk], [outsider], objs, [ring1]))  # key not in that ring
    assert refused(lambda: cls.prove_multi(alphas[:1], ads[:1], sks[:1], pks[:1], objs, [len(objs)]))  # index out of range
    assert refused(lambda: cls.prove_multi(alphas[:2], ads[:2], sks[:2], pks[:2], objs, index[:1]))  # one index per item
    assert cls.prove_multi([], [], [], [], objs, []) == []


# ---- 5. errors ---------------------------------------------------------------------------------------------------------------------


def errors(ctx, srs, other_srs, other_ctx, other_ctx_srs) -> None:
    """DR_EINVAL / ValueError: an index out of range, rings on two dr_srs handles, SHA-512 and SHAKE128 rings mixed, a ring of another
    context, n_rings == 0 with items; n == 0 proves nothing and raises nothing."""
    rings, items = reference_rings()
    natives = build(srs, rings)
    it = items[:1]

    def refused(fn) -> bool:
        try:
            fn()
        except ValueError:
            return True
        return False

    assert prove_multi(natives, it)[1] == [0]
    out_of_range = [(len(natives),) + it[0][1:]]
    assert refused(lambda: prove_multi(natives, out_of_range))
    keys, params = rings[0]
    twin = native_ring(other_srs, keys, params)
    assert refused(lambda: prove_multi(natives + [twin], it))
    twin.close()
    shake = load(SUITES[1][1] + "_ring.json")[0]
    sring = native_ring(srs, split_keys(hx(shake, "ring_pks")), rp.Params(test_vectors=True, suite=SUITES[1][0]))
    assert refused(lambda: prove_multi(natives + [sring], it))
    assert refused(lambda: prove_multi([sring] + natives, [(1,) + it[0][1:]]))
    sring.close()
    foreign = native_ring(other_ctx_srs, keys, params)
    assert refused(lambda: prove_multi(natives + [foreign], it))
    assert refused(lambda: prove_multi([foreign] + natives, [(1,) + it[0][1:]]))
    foreign.close()
    # raw ABI: n_rings == 0 with one item, an index out of range; n == 0 without rings
    lib = ctx.library.lib
    pk = _native.NativeRing.pack_prove_inputs([it[0][1]], [it[0][2]], [it[0][3]], [it[0][5]], ring_index=[0])
    args = _native.NativeRing._packed_args(pk, 0, 1)
    assert lib.dr_ring_prove_multi(ctx.handle, None, 0, pk["ring"], 1, *args) == _native.DR_EINVAL
    handles = (_native.c_void_p * 1)(natives[0].handle)
    pk_bad = _native.NativeRing.pack_prove_inputs([it[0][1]], [it[0][2]], [it[0][3]], [it[0][5]], ring_index=[1])
    assert lib.dr_ring_prove_multi(ctx.handle, handles, 1, pk_bad["ring"], 1, *_native.NativeRing._packed_args(pk_bad, 0, 1)) == _native.DR_EINVAL
    assert lib.dr_ring_prove_multi(ctx.handle, None, 0, None, 0, *[None] * 10) == _native.DR_OK
    assert _native.NativeRing.prove_multi(natives, [], [], [], [], []) == ([], [])
    assert _native.NativeRing.prove_multi([], [], [], [], [], []) == ([], [])
    for r in natives:
        r.close()


# ---- 6. an EnginePool gives the bytes of one engine ------------------------------------------------------------------------------


def pool_matches_one_engine(api, engine, pool, with_2048: bool = False) -> None:
    """RingVRF.prove_multi over rings built on a two-device EnginePool (contiguous shards, each device proving against its own
    replicas) gives the bytes of the same rings on one engine; rings of two engines are refused."""
    cls = api.RingVRF[api.Bandersnatch]
    rings, _ = reference_rings(with_2048)
    one = api_rings(api, engine, rings)
    many = api_rings(api, pool, rings)
    items = shuffled_batch(rings, 2, 17, with_2048)
    args = ([it[1] for it in items], [it[2] for it in items], [it[3] for it in items], [it[4] for it in items])
    index = [it[0] for it in items]
    zk = zk_of(items)
    want = cls.prove_multi(*args, one, index, zk_rows=zk, as_bytes=True)
    assert cls.prove_multi(*args, many, index, zk_rows=zk, as_bytes=True) == want
    try:
        cls.prove_multi(*args, [one[0]] + many[1:], index, zk_rows=zk, as_bytes=True)
    except ValueError:
        pass
    else:
        raise AssertionError("rings of an Engine and an EnginePool were accepted in one call")
    for r in one + many:
        r.native.close()


# ---- 8. full size (GPU) ----------------------------------------------------------------------------------------------------------


def eight_rings_1023(srs, per: int = 512):
    """Eight distinct rings of 1023 keys (seeded secrets; ring r > 0 replaces key 1000) and `per` items on each, interleaved:
    -> (ring key lists, params, items)."""
    from oracle import bandersnatch as bs
    from oracle import transcript as otr
    from tests.helpers import bench_ring_keys, seed

    params = rp.Params.from_ring_size(1023)
    pk, sk, base = bench_ring_keys(1023)
    keys = []
    for r in range(8):
        k = list(base)
        if r:
            k[1000] = otr.secret_from_seed(bs.SHA512, seed("multi-ring-test", r))[0]
        keys.append(k)
    rng = random.Random(5)
    items = []
    for j in range(per):
        for r in range(8):
            items.append((r, b"multi-%d-" % r + le64(j), b"multi-ad-%d-" % r + le64(j), sk, pk, 3, [rng.randrange(fr.R) for _ in range(12)], None))
    return keys, params, items

