"""Ring roots from keys, and their updates (dr_ring_roots_from_keys / dr_ring_root_update, RingRoot.from_keys / from_key_sets /
update): cases shared by the CPU (emulation build) and GPU (CUDA build) suites.

Every root is pinned by a root the reference published, or by dr_ring_root of dr_ring_create on the same keys, params and SRS G1
points.  An update is also checked against from_keys of the updated key list, and its inverse must give back the bytes it started
from."""

from __future__ import annotations

import random

from dot_ring_b200 import _native
from dot_ring_b200.srs import read_srs_file
from oracle import bandersnatch as bs
from oracle import bls12_381 as bls
from oracle import ring_proof as rp
from tests import adversarial_cases as adv
from tests.helpers import bench_ring_keys, hx, load, ring_proof_bytes, split_keys
from tests.msm_cases import TAU
from tests.ring_fixtures import native_ring
from tests.verify_cases import SUITES

NULL = b"\xff" * 32  # y >= p: never decodes, so the row holds the padding point


def root_params(params: rp.Params) -> _native.RingParamsStruct:
    s = params.suite
    return _native.make_ring_params(
        domain_size=params.domain_size, max_ring_size=params.max_ring_size, padding_rows=params.padding_rows, omega=params.omega,
        radix_omega=params.radix_omega, seed=s.accumulator_base, blinding_base=s.blinding_base, padding_point=s.padding_point,
        generator=bs.GENERATOR, suite_id=s.suite_id, h2c_dst=s.dst, hash_name=s.hash_name,
    )  # fmt: skip


def root_srs(ctx, n: int, g1_be96: bytes | None = None) -> _native.NativeSrs:
    """The first n points of an SRS (default: the bundled one) with the table Engine.root_srs builds (4-bit windows, GLV halves)."""
    raw = read_srs_file(None, None)
    return _native.NativeSrs(ctx, (g1_be96 if g1_be96 is not None else raw.g1_be96)[: 96 * n], raw.g2_be192, 4, 0, True)


def synthetic_g1(ctx, n: int) -> bytes:
    """tau^i * G, i < n (tests/extended_domain.py), for domains whose 3N + 1 points the bundled SRS does not hold."""
    return ctx.g1_synthetic_srs(TAU, 0, n)


def synthetic_ring_srs(ctx, n: int, window_bits: int) -> _native.NativeSrs:
    g2_gen = rp.load_srs().g2[0]
    g2 = bls.g2_serialize(g2_gen) + bls.g2_serialize(bls.g2_mul(g2_gen, TAU))
    return _native.NativeSrs(ctx, synthetic_g1(ctx, n), g2, window_bits)


def roots(srs, params: rp.Params, key_sets) -> list[bytes]:
    return _native.ring_roots_from_keys(srs, root_params(params), [list(k) for k in key_sets])


def update(srs, params: rp.Params, root: bytes, rows, new, old=None) -> bytes:
    return _native.ring_root_update(srs, root_params(params), root, list(rows), list(new), None if old is None else list(old))


def created_root(ring_srs, keys, params: rp.Params) -> bytes:
    """dr_ring_root of dr_ring_create: the root the prover's ring has."""
    ring = native_ring(ring_srs, list(keys), params)
    try:
        return ring.root()
    finally:
        ring.close()


def fresh_keys(ctx, n: int, seed: int) -> list[bytes]:
    """n valid public keys: multiples of the generator, computed on the device."""
    if not n:
        return []
    rng = random.Random(seed)
    return ctx.te_mul([bs.point_to_string(bs.GENERATOR)], [rng.randrange(1, bs.N) for _ in range(n)])


def refused(fn) -> bool:
    try:
        fn()
    except ValueError:
        return True
    return False


# ---- 1. roots the reference published --------------------------------------------------------------------------------------


def reference_pins(srs_for) -> None:
    """The ark-vrf ring vectors of both suites (ring_pks -> ring_pks_com, one call per suite) and the four rings of
    small_ring_reference.json (max_ring_size 100, 100 and 1 at N = 512, 6 at N = 2048).  srs_for(N) gives a root SRS."""
    for suite, prefix in SUITES:
        params = rp.Params(test_vectors=True, suite=suite)
        vecs = load(prefix + "_ring.json")
        assert roots(srs_for(params.domain_size), params, [split_keys(hx(v, "ring_pks")) for v in vecs]) == [hx(v, "ring_pks_com") for v in vecs], prefix
    for e in load("small_ring_reference.json"):
        params = rp.Params(domain_size=e["domain_size"], max_ring_size=e["max_ring_size"], test_vectors=e["test_vectors"])
        keys = [bytes.fromhex(k) for k in e["keys"]]
        assert roots(srs_for(params.domain_size), params, [keys]) == [bytes.fromhex(e["ring_root"])], (e["domain_size"], e["max_ring_size"])


def ring1023_pin(srs) -> None:
    ref = load("ring1023_reference.json")
    params = rp.Params.from_ring_size(1023)
    assert params.domain_size == ref["domain_size"] == 2048
    _, _, keys = bench_ring_keys(1023)
    assert roots(srs, params, [keys]) == [bytes.fromhex(ref["ring_root"])]


# ---- 2. byte-equal to dr_ring_create ----------------------------------------------------------------------------------------


def key_cases(ctx, params: rp.Params, seed: int = 0) -> list[tuple[str, list[bytes]]]:
    """(name, keys): no key, one, max_ring_size keys, undecodable keys, the identity, every te_mutations value (off-subgroup,
    small-order, sign-flipped ...) between valid keys, and duplicates."""
    base = fresh_keys(ctx, params.max_ring_size, seed)
    mutated = []
    for i, (_, value) in enumerate(adv.te_mutations(base[0])):
        mutated += [base[i + 1], value]
    identity = bs.point_to_string(bs.IDENTITY)
    return [
        ("empty", []),
        ("one", base[:1]),
        ("full", base),
        ("undecodable", [base[0], NULL, base[1], bytes(32), base[2]]),
        ("identity", [identity, base[0], identity]),
        ("te_mutations", mutated),
        ("duplicates", [base[0], base[1], base[0], base[0], base[2], base[1]]),
    ]


def same_as_ring_create(ctx, srs, ring_srs, params: rp.Params, seed: int = 0) -> None:
    """Every key case in one from_keys call, each root byte-equal to dr_ring_root of dr_ring_create on the same keys."""
    cases = key_cases(ctx, params, seed)
    got = roots(srs, params, [keys for _, keys in cases])
    for (name, keys), root in zip(cases, got):
        assert root == created_root(ring_srs, keys, params), (params.domain_size, params.suite.name, name)


def large_domain(ctx, n_keys: int, domain: int, ring_window_bits: int, seed: int = 3) -> None:
    """A domain above the reference's 4096 over a synthetic SRS: from_keys over its first N points against dr_ring_create over
    its first 3N + 1 points (narrow windows), then an update against the ring rebuilt from the changed keys."""
    params = rp.Params(domain_size=domain, max_ring_size=domain - rp.SCALAR_BITS - 4, max_domain_size=max(domain, 4096))
    ring_srs = synthetic_ring_srs(ctx, 3 * domain + 1, ring_window_bits)
    srs = root_srs(ctx, domain, synthetic_g1(ctx, domain))
    try:
        keys = fresh_keys(ctx, n_keys, seed)
        root = roots(srs, params, [keys])[0]
        assert root == created_root(ring_srs, keys, params)
        new = fresh_keys(ctx, 2, seed + 1)
        rows = [n_keys // 2, n_keys]  # a replacement and an append (the old key of a padding row: any key that does not decode)
        changed = keys[: rows[0]] + [new[0]] + keys[rows[0] + 1 :] + [new[1]]
        root2 = update(srs, params, root, rows, new, [keys[rows[0]], NULL])
        assert root2 == created_root(ring_srs, changed, params) == roots(srs, params, [changed])[0]
    finally:
        srs.close()
        ring_srs.close()


# ---- 3. batching ------------------------------------------------------------------------------------------------------------


def batching(ctx, srs, ring_srs, params: rp.Params, counts=(3, 0, 1, 7, 0, 2), seed: int = 100) -> None:
    """K rings with different key counts (0 included) give the same bytes in one call, in K calls and from K dr_ring_create."""
    sets = [fresh_keys(ctx, c, seed + i) for i, c in enumerate(counts)]
    one_call = roots(srs, params, sets)
    assert one_call == [roots(srs, params, [keys])[0] for keys in sets]
    assert one_call == [created_root(ring_srs, keys, params) for keys in sets]
    assert roots(srs, params, []) == []


# ---- 4. updates -------------------------------------------------------------------------------------------------------------


def update_walk(ctx, srs, ring_srs, params: rp.Params, steps: int, seed: int, check_created_every: int = 1) -> None:
    """A seeded sequence of appends into padding rows, replacements, nullings, restores and multi-row updates.  After every step the
    root equals from_keys of the current key list (all states in one call at the end) and, every `check_created_every` steps,
    dr_ring_root; the inverse update gives back the previous bytes."""
    rng = random.Random(seed)
    cap = params.max_ring_size
    supply = iter(fresh_keys(ctx, 8 * steps + 8, seed))
    identity = bs.point_to_string(bs.IDENTITY)
    # encodings that put the padding point in a row: undecodable, the identity, off-subgroup and small-order points
    nulls = [v for v in [NULL, identity, bytes(32)] + [v for _, v in adv.te_mutations(next(supply))] if ctx.te_decode([v])[0] is None]
    keys = [next(supply) for _ in range(3)]  # the key list; rows from len(keys) on hold padding
    nulled: dict[int, bytes] = {}  # row -> the key it held before it was nulled
    root = roots(srs, params, [keys])[0]
    states, seen = [(list(keys), root)], set()
    for step in range(steps):
        kinds = ["append", "replace", "null", "restore", "multi"]
        kind = kinds[step] if step < len(kinds) else rng.choice(kinds)
        live = [r for r in range(len(keys)) if r not in nulled]
        if kind == "restore" and not nulled:
            kind = "null"
        if kind in ("replace", "null", "multi") and len(live) < 2:
            kind = "append" if len(keys) < cap else "restore"
        if kind == "append" and len(keys) >= cap:
            kind = "replace" if live else "restore"
        seen.add(kind)
        if kind == "append":
            a = min(rng.randint(1, 3), cap - len(keys))
            rows, old, new = list(range(len(keys), len(keys) + a)), None, [next(supply) for _ in range(a)]
        elif kind == "replace":
            rows = rng.sample(live, min(len(live), rng.randint(1, 2)))
            old, new = [keys[r] for r in rows], [next(supply) for _ in rows]
        elif kind == "null":
            rows = rng.sample(live, 1)
            old, new = [keys[rows[0]]], [rng.choice(nulls)]
        elif kind == "restore":
            rows = [rng.choice(sorted(nulled))]
            old, new = [keys[rows[0]]], [nulled[rows[0]]]
        else:  # several rows at once: replacements, a nulling and, while there is room, an append with an undecodable old key
            rows = rng.sample(live, min(len(live), rng.randint(2, 4)))
            old = [keys[r] for r in rows]
            new = [next(supply) for _ in rows[:-1]] + [rng.choice(nulls)]
            if len(keys) < cap:
                rows, old, new = rows + [len(keys)], old + [rng.choice(nulls)], new + [next(supply)]
        new_root = update(srs, params, root, rows, new, old)
        assert update(srs, params, new_root, rows, old if old is not None else [NULL] * len(rows), new) == root, (step, kind)
        for r, k_old, k_new in zip(rows, old if old is not None else [None] * len(rows), new):
            if r == len(keys):
                keys.append(k_new)
            else:
                keys[r] = k_new
            if kind == "restore":
                nulled.pop(r)
            elif k_new in nulls:
                nulled.setdefault(r, k_old)
            else:
                nulled.pop(r, None)
        if step % check_created_every == 0 or step == steps - 1:
            assert new_root == created_root(ring_srs, keys, params), (step, kind)
        states.append((list(keys), new_root))
        root = new_root
    assert seen == {"append", "replace", "null", "restore", "multi"}
    assert roots(srs, params, [k for k, _ in states]) == [r for _, r in states]


# ---- 5. errors ---------------------------------------------------------------------------------------------------------------


def abi_errors(ctx, other_ctx, srs, params: rp.Params) -> None:
    """DR_EINVAL for each rejected input, from both functions where it applies; DR_OK for empty calls."""
    N = params.domain_size
    keys = fresh_keys(ctx, 3, 7)
    good = roots(srs, params, [keys])[0]
    both = lambda p, s=srs: (  # noqa: E731
        refused(lambda: _native.ring_roots_from_keys(s, p, [keys])) and refused(lambda: _native.ring_root_update(s, p, good, [0], keys[:1], keys[:1]))
    )
    for field, value in (("domain_size", 256), ("domain_size", 1000), ("domain_size", 1 << 17), ("padding_rows", 3), ("max_ring_size", N - rp.SCALAR_BITS - 3)):
        p = root_params(params)
        setattr(p, field, value)
        assert both(p), (field, value)
    for omega in (params.omega * params.omega % bls.R, 1, params.omega + bls.R):  # not primitive, not canonical
        p = root_params(params)
        p.omega[:] = list((omega % (1 << 256)).to_bytes(32, "little"))
        assert both(p), omega
    p = root_params(params)
    p.padding_point[:] = list(b"\x05" * 64)  # not on the curve
    assert both(p)
    # more keys than max_ring_size
    assert refused(lambda: roots(srs, params, [[], fresh_keys(ctx, params.max_ring_size + 1, 8)]))
    # an SRS of N - 1 points; an SRS of another context
    short = root_srs(ctx, N - 1)
    assert both(root_params(params), short)
    short.close()
    lib, p, ref = ctx.library.lib, root_params(params), _native.ctypes.byref
    out = _native.ctypes.create_string_buffer(144)
    rows = (_native.c_uint32 * 1)(0)
    foreign = root_srs(other_ctx, N)
    assert lib.dr_ring_roots_from_keys(ctx.handle, foreign.handle, ref(p), 1, keys[0], (_native.c_uint32 * 1)(1), out) == _native.DR_EINVAL
    assert lib.dr_ring_root_update(ctx.handle, foreign.handle, ref(p), good, 1, rows, None, keys[0], out) == _native.DR_EINVAL
    assert lib.dr_ring_roots_from_keys(other_ctx.handle, foreign.handle, ref(p), 1, keys[0], (_native.c_uint32 * 1)(1), out) == _native.DR_OK
    foreign.close()
    # rows: out of range, twice in one update
    assert refused(lambda: update(srs, params, good, [params.max_ring_size], keys[:1]))
    assert refused(lambda: update(srs, params, good, [1, 1], keys[:2]))
    assert refused(lambda: update(srs, params, good, [0, 5, 0], keys))
    # a root that does not decode: refused exactly where RingRoot.decode raises, each commitment mutated
    for j in range(3):
        field = good[48 * j : 48 * j + 48]
        for name, value in adv.g1_mutations(field, good[48 * ((j + 1) % 3) : 48 * ((j + 1) % 3) + 48]):
            mutated = good[: 48 * j] + value + good[48 * j + 48 :]
            try:
                rp.decode_ring_root(mutated)
            except ValueError:
                assert refused(lambda: update(srs, params, mutated, [4], keys[:1])), (j, name)
                continue
            if j < 2:  # decodes: the update is linear whatever the point, and its inverse restores the bytes
                there = update(srs, params, mutated, [4], keys[:1])
                assert update(srs, params, there, [4], [NULL], keys[:1]) == mutated, (j, name)
            else:  # any other C_s is not this params' C_s
                assert (value == field) != refused(lambda: update(srs, params, mutated, [4], keys[:1])), name
    # a root built for other params (C_s differs), or over another SRS
    other = rp.Params(domain_size=N, max_ring_size=params.max_ring_size - 1, test_vectors=True, suite=params.suite)
    assert refused(lambda: update(srs, params, roots(srs, other, [keys])[0], [0], keys[:1]))
    foreign = root_srs(ctx, N, synthetic_g1(ctx, N))
    assert refused(lambda: update(srs, params, roots(foreign, params, [keys])[0], [0], keys[:1]))
    foreign.close()
    # null pointers
    assert lib.dr_ring_root_update(ctx.handle, srs.handle, ref(p), good, 1, rows, None, None, out) == _native.DR_EINVAL
    assert lib.dr_ring_roots_from_keys(ctx.handle, srs.handle, ref(p), 1, None, (_native.c_uint32 * 1)(2), out) == _native.DR_EINVAL
    # empty calls; n == 0 copies the root, and out may be the input
    assert lib.dr_ring_roots_from_keys(ctx.handle, srs.handle, ref(p), 0, None, None, None) == _native.DR_OK
    assert update(srs, params, good, [], []) == good
    inout = _native.ctypes.create_string_buffer(good, 144)
    assert lib.dr_ring_root_update(ctx.handle, srs.handle, ref(p), inout, 1, rows, keys[0], keys[1], inout) == _native.DR_OK
    assert inout.raw == update(srs, params, good, [0], keys[1:2], keys[:1]) != good


def api_errors(api, engine) -> None:
    """The ValueErrors RingRoot.from_keys / update raise where the ABI returns DR_EINVAL, and a root left unchanged by update."""
    params = api.RingProofParams(test_vectors=True)
    v = load(SUITES[0][1] + "_ring.json")[0]
    keys = split_keys(hx(v, "ring_pks"))
    assert refused(lambda: api.RingRoot.from_keys(keys * 40, params, engine))
    root = api.RingRoot.from_keys(keys, params, engine)
    before = root.fixed_commitments()
    assert refused(lambda: root.update([params.max_ring_size], keys[:1]))
    assert refused(lambda: root.update([1, 1], keys[:2]))
    assert refused(lambda: root.update([1], keys[:2]))
    small = api.RingProofParams(domain_size=512, max_ring_size=100, test_vectors=True)
    foreign = api.RingRoot.from_keys(keys, small, engine)
    assert refused(lambda: api.RingRoot(foreign.px, foreign.py, foreign.s, params, engine).update([0], keys[:1]))
    assert refused(lambda: root.update([0], [keys[0]], [keys[1], keys[2]]))
    assert root.fixed_commitments() == before
    # max_ring_size keys are fine, one more is not
    assert api.RingRoot.from_key_sets([keys * 31 + keys[:7]], params, engine)[0].params is params
    assert refused(lambda: api.RingRoot.from_key_sets([keys, keys * 32], params, engine))


# ---- 6. the Python API ------------------------------------------------------------------------------------------------------


def api_semantics(api, engine) -> None:
    """from_keys equals from_ring of Ring(keys) with default and explicit params, keys of the wrong length included; update of a
    decoded root; from_key_sets equals from_keys one by one."""
    v = load(SUITES[0][1] + "_ring.json")[0]
    keys = split_keys(hx(v, "ring_pks"))
    enc = lambda r: engine.ctx.g1_compress(b"".join(r.fixed_commitments()))  # noqa: E731
    params = api.RingProofParams(test_vectors=True)
    root = api.RingRoot.from_keys(keys, params, engine)
    assert enc(root) == hx(v, "ring_pks_com") and root.params is params
    odd = [keys[0], b"short", keys[1], b"x" * 33, keys[2]]
    assert enc(api.RingRoot.from_keys(odd, params, engine)) == enc(api.RingRoot.from_ring(api.Ring(odd, params, engine), params))
    default = api.RingRoot.from_keys(keys, engine=engine)
    ring = api.Ring(keys, engine=engine)
    assert default.params.domain_size == ring.params.domain_size and enc(default) == enc(api.RingRoot.from_ring(ring))
    # update: a decoded root, keys of the wrong length mapped as in Ring, self unchanged
    decoded = api.RingRoot.decode(hx(v, "ring_pks_com"), params)
    changed = list(keys)
    changed[5] = b"short"
    upd = decoded.update([5], [b"short"], [keys[5]])
    assert enc(upd) == enc(api.RingRoot.from_keys(changed, params, engine)) and enc(decoded) == hx(v, "ring_pks_com")
    assert enc(upd.update([5], [keys[5]], [b"short"])) == hx(v, "ring_pks_com")
    appended = upd.update([8, 9], keys[:2])
    assert enc(appended) == enc(api.RingRoot.from_keys(changed + keys[:2], params, engine))
    sets = [keys, [], keys[:3], odd]
    assert [enc(r) for r in api.RingRoot.from_key_sets(sets, params, engine)] == [enc(api.RingRoot.from_keys(s, params, engine)) for s in sets]
    assert api.RingRoot.from_key_sets([], params, engine) == []


def no_window_table(api, engine) -> None:
    """On a fresh engine: from_keys, update and a RingVerifier check of an ark-vrf proof against that root; the prover's window
    table is never built."""
    assert engine._srs is None
    v = load(SUITES[0][1] + "_ring.json")[0]
    keys = split_keys(hx(v, "ring_pks"))
    params = api.RingProofParams(test_vectors=True)
    root = api.RingRoot.from_keys(keys, params, engine)
    nulled = root.update([2], [NULL], [keys[2]])
    back = nulled.update([2], [keys[2]], [NULL])
    assert back.fixed_commitments() == root.fixed_commitments() != nulled.fixed_commitments()
    verifier = api.RingVerifier([back], engine)
    proof, alpha, ad = ring_proof_bytes(v), hx(v, "alpha"), hx(v, "ad")
    assert verifier.verify(proof, alpha, ad) and verifier.batch_verify([proof], [alpha], [ad])
    assert not verifier.verify(proof, alpha, ad + b"x")
    verifier.close()
    assert api.RingVerifier([nulled], engine).verify_batch([proof], [alpha], [ad]) == [0]
    assert engine._srs is None and params.domain_size in engine._root_srs


def pool_matches_one_engine(api, engine, pool) -> None:
    """An EnginePool gives the bytes of one engine, for from_key_sets, from_keys and update."""
    v = load(SUITES[0][1] + "_ring.json")[0]
    keys = split_keys(hx(v, "ring_pks"))
    params = api.RingProofParams(test_vectors=True)
    sets = [keys, keys[:3], [], keys[::-1]]
    one = api.RingRoot.from_key_sets(sets, params, engine)
    many = api.RingRoot.from_key_sets(sets, params, pool)
    assert [r.fixed_commitments() for r in one] == [r.fixed_commitments() for r in many]
    assert api.RingRoot.from_keys(keys, params, pool).fixed_commitments() == one[0].fixed_commitments()
    a = one[1].update([3, 0], [keys[4], NULL], [NULL, keys[0]])
    b = many[1].update([3, 0], [keys[4], NULL], [NULL, keys[0]])
    assert a.fixed_commitments() == b.fixed_commitments() and b.engine is pool
    assert all(e._srs is None for e in pool.engines)
