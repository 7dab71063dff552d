"""Keyless, multi-ring Ring VRF verification (dr_ring_verifier_create / dr_ring_verify_multi, dot_ring_b200.RingVerifier): cases
shared by the CPU (emulation build) and GPU (CUDA build) suites.

A verifier is built from a 144-byte ring root alone.  Every verdict is pinned by the reference's vectors, by dr_ring_verify_batch
on the same bytes and coefficients, or by the CPU oracle run on the root bytes (rp.decode_ring_root plus a transcript prefix over
the decoded commitments): per item, Pedersen-ok and rp.batch_verify_linear of that item's two openings; aggregated,
rp.batch_verify_linear over the union of the batch's openings with the same coefficients."""

from __future__ import annotations

import random

from dot_ring_b200 import _native
from dot_ring_b200.srs import read_srs_file
from oracle import bandersnatch as bs
from oracle import bls12_381 as bls
from oracle import ring_proof as rp
from oracle import transcript as otr
from oracle import vrf as ovrf
from tests import adversarial_cases as adv
from tests.helpers import hx, load, ring_proof_bytes, split_keys
from tests.ring_fixtures import native_ring
from tests.verify_cases import SUITES

R = bls.R


def srs_head():
    """([1]_1 as 96 bytes, [1]_2 | [tau]_2 as 384 bytes) of the bundled SRS: all a verifier takes from it."""
    raw = read_srs_file(None, 1)
    return raw.g1_be96[:96], raw.g2_be192


def make_verifier(ctx, root: bytes, params: rp.Params) -> _native.NativeRingVerifier:
    s = params.suite
    g1_0, g2 = srs_head()
    return _native.NativeRingVerifier(
        ctx, root, g1_0, g2, domain_size=params.domain_size, omega=params.omega, seed=s.accumulator_base, blinding_base=s.blinding_base,
        generator=bs.GENERATOR, suite_id=s.suite_id, h2c_dst=s.dst, hash_name=s.hash_name,
    )  # fmt: skip


def multi(verifiers, index, alphas, ads, proofs, coeffs, aggregate=False, msm_threshold=None):
    """verify_multi, optionally through the two-MSM route (dr_ring_verify_set_msm_threshold), restoring the default."""
    lib = verifiers[0].ctx.library.lib
    if msm_threshold is not None:
        lib.dr_ring_verify_set_msm_threshold(msm_threshold)
    try:
        return _native.NativeRingVerifier.verify_multi(verifiers, index, alphas, ads, proofs, coeffs, aggregate)
    finally:
        if msm_threshold is not None:
            lib.dr_ring_verify_set_msm_threshold(8192)


def both_routes(verifiers, index, alphas, ads, proofs, coeffs):
    """(verdicts, all_ok) of the aggregated check through the 13-multiplication route and the two-MSM route; they must agree."""
    a = multi(verifiers, index, alphas, ads, proofs, coeffs, aggregate=True)
    b = multi(verifiers, index, alphas, ads, proofs, coeffs, aggregate=True, msm_threshold=1)
    assert a == b
    return a


class RootOracle:
    """The oracle's ring verifier for one root, from the root bytes alone."""

    def __init__(self, root: bytes, params: rp.Params):
        self.params = params
        self.srs = rp.load_srs()
        self.fixed = tuple(rp.decode_ring_root(root))
        self.prefix = otr.RingTranscript(params.suite.suite_id)
        self.prefix.absorb_labeled(b"vk", rp.srs_vk_prefix(self.srs) + b"".join(bls.g1_serialize(c) for c in self.fixed))

    def parts(self, proof: bytes, alpha: bytes, ad: bytes):
        """(status, linear verifications): 2 = decode raises, 0 = Pedersen part rejected, 1 = accepted."""
        try:
            p = ovrf.RingVrfProof.decode(proof)
        except ValueError:
            return 2, None
        ok = ovrf.pedersen_verify(self.params.suite, p.pedersen, alpha, ad)
        return int(ok), rp.linear_verifications(self.params, self.fixed, self.prefix, p.pedersen.blinded_pk, p.ring)


def oracle_verdicts(oracles, index, alphas, ads, proofs, coeffs):
    """(per-item verdicts, per-item status, aggregated result) of the oracle for a batch spanning several roots."""
    parts = [oracles[k].parts(p, a, d) for k, p, a, d in zip(index, proofs, alphas, ads)]
    srs = oracles[0].srs
    verdicts = [st if st != 1 else int(rp.batch_verify_linear(srs, lin, coeffs[2 * i : 2 * i + 2])) for i, (st, lin) in enumerate(parts)]
    status = [st for st, _ in parts]
    agg = all(st == 1 for st in status) and bool(rp.batch_verify_linear(srs, [v for _, lin in parts for v in lin], list(coeffs)))
    return verdicts, status, agg


def independent(n: int, seed: int) -> list[int]:
    rng = random.Random(seed)
    return [v for _ in range(n) for v in (1, rng.randrange(1, R))]


# ---- 1. keyless verification pinned by the reference's vectors -------------------------------------------------------------


def ark_ring_vectors(prefix: str):
    """(root, alpha, ad, proof) of every ark-vrf ring vector of one suite."""
    return [(hx(v, "ring_pks_com"), hx(v, "alpha"), hx(v, "ad"), ring_proof_bytes(v)) for v in load(prefix + "_ring.json")]


def keyless_reference_vectors(ctx) -> None:
    for suite, prefix in SUITES:
        params = rp.Params(test_vectors=True, suite=suite)
        for root, alpha, ad, proof in ark_ring_vectors(prefix):
            v = make_verifier(ctx, root, params)
            got, ok = multi([v], [0, 0, 0], [alpha, alpha, alpha + b"x"], [ad, ad + b"x", ad], [proof] * 3, independent(3, 1))
            assert got == [1, 0, 0] and not ok, prefix
            v.close()
    # the seven SHA-512 vectors in one batch, each against its own ring (six distinct roots)
    params = rp.Params(test_vectors=True)
    vecs = ark_ring_vectors(SUITES[0][1])
    roots = list(dict.fromkeys(r for r, _, _, _ in vecs))
    assert len(vecs) == 7 and len(roots) == 6
    verifiers = [make_verifier(ctx, r, params) for r in roots]
    index = [roots.index(r) for r, _, _, _ in vecs]
    alphas, ads, proofs = [a for _, a, _, _ in vecs], [d for _, _, d, _ in vecs], [p for _, _, _, p in vecs]
    n = len(vecs)
    assert multi(verifiers, index, alphas, ads, proofs, independent(n, 2)) == ([1] * n, True)
    assert both_routes(verifiers, index, alphas, ads, proofs, adv.coeffs_random(n, 3)) == ([1] * n, True)
    # every proof against a ring that is not its own
    rotated = [(k + 1) % len(roots) for k in index]
    assert multi(verifiers, rotated, alphas, ads, proofs, independent(n, 4)) == ([0] * n, False)
    assert both_routes(verifiers, rotated, alphas, ads, proofs, adv.coeffs_random(n, 5)) == ([1] * n, False)
    for v in verifiers:
        v.close()


# ---- 2. mixed domains ----------------------------------------------------------------------------------------------------


def mixed_domain_items(with_ring1023: bool = False):
    """[(root, params, alpha, ad, proof)]: the N = 512 / 2048 small-ring fixtures, the SHA-512 ark-vrf rings and, on request, the six
    ring-1023 reference proofs (N = 2048)."""
    items = []
    for e in load("small_ring_reference.json"):
        params = rp.Params(domain_size=e["domain_size"], max_ring_size=e["max_ring_size"], test_vectors=e["test_vectors"])
        items.append((bytes.fromhex(e["ring_root"]), params, bytes.fromhex(e["alpha"]), bytes.fromhex(e["ad"]), bytes.fromhex(e["proof"])))
    params = rp.Params(test_vectors=True)
    items += [(r, params, a, d, p) for r, a, d, p in ark_ring_vectors(SUITES[0][1])]
    if with_ring1023:
        ref = load("ring1023_reference.json")
        params = rp.Params.from_ring_size(1023)
        assert params.domain_size == ref["domain_size"]
        for e in ref["proofs_test_vectors"] + ref["proofs_blinded"]:
            items.append((bytes.fromhex(ref["ring_root"]), params, bytes.fromhex(e["alpha"]), bytes.fromhex(e["ad"]), bytes.fromhex(e["proof"])))
    return items


def build_batch(ctx, items):
    """One verifier per distinct (root, domain); -> (verifiers, index, alphas, ads, proofs)."""
    keys = list(dict.fromkeys((r, p.domain_size, p.max_ring_size) for r, p, _, _, _ in items))
    params = {(r, p.domain_size, p.max_ring_size): p for r, p, _, _, _ in items}
    verifiers = [make_verifier(ctx, k[0], params[k]) for k in keys]
    index = [keys.index((r, p.domain_size, p.max_ring_size)) for r, p, _, _, _ in items]
    return verifiers, index, [i[2] for i in items], [i[3] for i in items], [i[4] for i in items]


def mixed_domains(ctx, with_ring1023: bool = False) -> None:
    items = mixed_domain_items(with_ring1023)
    assert len({p.domain_size for _, p, _, _, _ in items}) >= 2
    verifiers, index, alphas, ads, proofs = build_batch(ctx, items)
    n = len(items)
    assert multi(verifiers, index, alphas, ads, proofs, independent(n, 6)) == ([1] * n, True)
    assert both_routes(verifiers, index, alphas, ads, proofs, adv.coeffs_random(n, 7)) == ([1] * n, True)
    for v in verifiers:
        v.close()


# ---- 3. same verdicts as the keyed path -------------------------------------------------------------------------------------


def same_as_keyed(ctx, srs, one_per_type: bool = True, fold_sample: int | None = None) -> None:
    """A verifier from dr_ring_root of a ring against dr_ring_verify_batch on that ring: same bytes, same coefficients, every
    ring_mutants proof per item and aggregated, and each decodable mutant folded between two valid proofs (both routes)."""
    _, keys, alpha, ad, proof = adv._ring_vector(SUITES[0][1])
    params = rp.Params(test_vectors=True)
    ring = native_ring(srs, keys, params)
    v = make_verifier(ctx, ring.root(), params)
    mutants = [m for _, m in adv.ring_mutants(proof, one_per_type=one_per_type)]
    n = len(mutants)
    co = independent(n, 8)
    assert multi([v], [0] * n, [alpha] * n, [ad] * n, mutants, co) == ring.verify_batch([alpha] * n, [ad] * n, mutants, co)
    co = adv.coeffs_random(n, 9)
    assert both_routes([v], [0] * n, [alpha] * n, [ad] * n, mutants, co) == ring.verify_batch([alpha] * n, [ad] * n, mutants, co, aggregate=True)
    oracle = RootOracle(ring.root(), params)
    folded = [m for m in mutants if oracle.parts(m, alpha, ad)[0] != 2]
    if fold_sample is not None:
        folded = folded[:fold_sample]
    lib = ring.ctx.library.lib
    for i, m in enumerate(folded):
        batch, co = [proof, m, proof], adv.coeffs_random(3, 200 + i)
        for threshold in (8192, 1):
            lib.dr_ring_verify_set_msm_threshold(threshold)
            try:
                want = ring.verify_batch([alpha] * 3, [ad] * 3, batch, co, aggregate=True)
            finally:
                lib.dr_ring_verify_set_msm_threshold(8192)
            assert multi([v], [0] * 3, [alpha] * 3, [ad] * 3, batch, co, aggregate=True, msm_threshold=threshold) == want, (i, threshold)
    v.close()
    ring.close()


# ---- 4. oracle parity across rings -------------------------------------------------------------------------------------------


def oracle_parity_across_rings(ctx, items=None) -> None:
    """A batch over several roots with honest items, a wrong ad, a wrong input, and proofs sent to another ring."""
    items = items if items is not None else mixed_domain_items()
    verifiers, index, alphas, ads, proofs = build_batch(ctx, items)
    roots = list(dict.fromkeys((r, p.domain_size, p.max_ring_size) for r, p, _, _, _ in items))
    params = {(r, p.domain_size, p.max_ring_size): p for r, p, _, _, _ in items}
    oracles = [RootOracle(k[0], params[k]) for k in roots]
    n = len(items)
    # honest items, then tampered copies of the first two
    index2 = index + [index[0], index[1], (index[0] + 1) % len(roots), (index[1] + 1) % len(roots)]
    alphas2 = alphas + [alphas[0], alphas[1] + b"!", alphas[0], alphas[1]]
    ads2 = ads + [ads[0] + b"!", ads[1], ads[0], ads[1]]
    proofs2 = proofs + [proofs[0], proofs[1], proofs[0], proofs[1]]
    for idx, al, dd, pr in ((index, alphas, ads, proofs), (index2, alphas2, ads2, proofs2)):
        m = len(pr)
        co = independent(m, 10 + m)
        want_v, _, _ = oracle_verdicts(oracles, idx, al, dd, pr, co)
        assert multi(verifiers, idx, al, dd, pr, co)[0] == want_v
        co = adv.coeffs_random(m, 20 + m)
        _, status, agg = oracle_verdicts(oracles, idx, al, dd, pr, co)
        assert both_routes(verifiers, idx, al, dd, pr, co) == (status, agg)
    assert n >= 2
    for v in verifiers:
        v.close()


# ---- 5. adversarial roots --------------------------------------------------------------------------------------------------


def adversarial_roots(ctx, sample: int | None = None) -> None:
    """Each commitment of a ring-8 root replaced by every g1_mutations value: creation fails exactly where rp.decode_ring_root
    raises; elsewhere per-item and aggregated verdicts (both routes) equal the oracle's.  The batch pairs the vector's own proof
    with a proof whose ad differs, each against the mutated root, and adds the honest proof against the honest root."""
    vecs = ark_ring_vectors(SUITES[0][1])
    root, alpha, ad, proof = vecs[0]
    params = rp.Params(test_vectors=True)
    honest = make_verifier(ctx, root, params)
    honest_oracle = RootOracle(root, params)
    reached_outside = 0
    cases = []
    for j in range(3):
        field = root[48 * j : 48 * j + 48]
        sibling = root[48 * ((j + 1) % 3) : 48 * ((j + 1) % 3) + 48]
        cases += [(j, name, root[: 48 * j] + value + root[48 * j + 48 :]) for name, value in adv.g1_mutations(field, sibling)]
    if sample is not None:
        keep = {"outside_g1", "plus_order3", "order3", "order11", "infinity", "generator", "x_off_curve", "x_ge_p"}
        cases = [c for c in cases if c[1] in keep][:sample]
    for j, name, mutated in cases:
        try:
            fixed = rp.decode_ring_root(mutated)
        except ValueError:
            fixed = None
        if fixed is None:
            try:
                make_verifier(ctx, mutated, params).close()
            except ValueError:
                continue
            raise AssertionError(f"verifier accepted a root the reference rejects: commitment {j}, {name}")
        reached_outside += any(c is not None and not adv.in_g1(c) for c in fixed)
        v = make_verifier(ctx, mutated, params)
        oracle = RootOracle(mutated, params)
        batch = ([1, 1, 0], [alpha, alpha, alpha], [ad, ad + b"?", ad], [proof, proof, proof])
        co = independent(3, 30 + j)
        want_v, _, _ = oracle_verdicts([honest_oracle, oracle], *batch, co)
        assert multi([honest, v], *batch, co)[0] == want_v, (j, name)
        co = adv.coeffs_random(3, 40 + j)
        _, status, agg = oracle_verdicts([honest_oracle, oracle], *batch, co)
        assert both_routes([honest, v], *batch, co) == (status, agg), (j, name)
        v.close()
    assert reached_outside, "no mutated root put a commitment outside G1 (the full-multiplication path)"
    honest.close()


# ---- 6. API edges ----------------------------------------------------------------------------------------------------------


def api_edges(api, engine) -> None:
    """RingVerifier: keyless verification from decoded roots, index and suite errors, empty batches, no window table built."""
    cls = api.RingVRF[api.Bandersnatch]
    vecs = ark_ring_vectors(SUITES[0][1])
    params = api.RingProofParams(test_vectors=True)
    roots = list(dict.fromkeys(r for r, _, _, _ in vecs))
    verifier = api.RingVerifier([api.RingRoot.decode(r, params) for r in roots], engine)
    index = [roots.index(r) for r, _, _, _ in vecs]
    alphas, ads, proofs = [a for _, a, _, _ in vecs], [d for _, _, d, _ in vecs], [p for _, _, _, p in vecs]
    assert verifier.verify_batch(proofs, alphas, ads, index) == [1] * len(vecs)
    assert verifier.batch_verify(proofs, alphas, ads, index)
    assert verifier.verify(cls.decode(proofs[0]), alphas[0], ads[0], index[0])
    assert not verifier.verify(proofs[0], alphas[0], ads[0] + b"x", index[0])
    assert not verifier.batch_verify(proofs, alphas, ads, [(k + 1) % len(roots) for k in index])
    assert verifier.verify_batch([], [], []) == [] and verifier.batch_verify([], [], [])
    try:
        verifier.verify_batch(proofs[:1], alphas[:1], ads[:1], [len(roots)])
    except ValueError:
        pass
    else:
        raise AssertionError("ring index out of range was accepted")
    assert not verifier.batch_verify(proofs[:1], alphas[:1], ads[:1], [len(roots)])
    # the default index is 0
    assert verifier.verify_batch(proofs[:1], alphas[:1], ads[:1]) == [1 if index[0] == 0 else 0]
    verifier.close()
    shake = load(SUITES[1][1] + "_ring.json")[0]
    sparams = api.RingProofParams(test_vectors=True, cv=api.Bandersnatch_SHAKE128)
    try:
        api.RingVerifier([api.RingRoot.decode(roots[0], params), api.RingRoot.decode(hx(shake, "ring_pks_com"), sparams)], engine)
    except ValueError:
        pass
    else:
        raise AssertionError("roots of two suites were accepted")
    # the SHAKE128 suite alone
    sv = api.RingVerifier([api.RingRoot.decode(hx(shake, "ring_pks_com"), sparams)], engine)
    assert sv.verify(ring_proof_bytes(shake), hx(shake, "alpha"), hx(shake, "ad"))
    sv.close()
    # a root from a ring, as RingRoot.from_ring gives it
    ring = api.Ring(split_keys(hx(load(SUITES[0][1] + "_ring.json")[0], "ring_pks")), params, engine)
    rv = api.RingVerifier([api.RingRoot.from_ring(ring, params)], engine)
    assert rv.verify(proofs[0], alphas[0], ads[0])
    rv.close()


def no_window_table(api, engine) -> None:
    """Building a RingVerifier and verifying leaves the engine's window table unbuilt."""
    assert engine._srs is None
    vecs = ark_ring_vectors(SUITES[0][1])
    params = api.RingProofParams(test_vectors=True)
    root, alpha, ad, proof = vecs[0]
    v = api.RingVerifier([api.RingRoot.decode(root, params)], engine)
    assert v.verify_batch([proof], [alpha], [ad]) == [1] and v.batch_verify([proof], [alpha], [ad])
    v.close()
    assert engine._srs is None


def errors_at_the_abi(ctx, other_ctx) -> None:
    """DR_EINVAL: verifiers of another context, of two suites, of two G2 pairs, an index out of range, a bad domain."""
    root, alpha, ad, proof = ark_ring_vectors(SUITES[0][1])[0]
    params = rp.Params(test_vectors=True)
    v = make_verifier(ctx, root, params)
    co = independent(1, 50)

    def refused(fn):
        try:
            fn()
        except ValueError:
            return True
        return False

    w = make_verifier(other_ctx, root, params)
    assert refused(lambda: multi([v, w], [0], [alpha], [ad], [proof], co))
    w.close()
    s = SUITES[1][0]
    shake_root = hx(load(SUITES[1][1] + "_ring.json")[0], "ring_pks_com")
    w = make_verifier(ctx, shake_root, rp.Params(test_vectors=True, suite=s))
    assert refused(lambda: multi([v, w], [0], [alpha], [ad], [proof], co))
    w.close()
    g1_0, g2 = srs_head()
    g2_other = g2[192:] + g2[:192]
    ps = params.suite
    w = _native.NativeRingVerifier(ctx, root, g1_0, g2_other, domain_size=512, omega=params.omega, seed=ps.accumulator_base, blinding_base=ps.blinding_base,
                                   generator=bs.GENERATOR, suite_id=ps.suite_id, h2c_dst=ps.dst, hash_name=ps.hash_name)
    assert refused(lambda: multi([v, w], [0], [alpha], [ad], [proof], co))
    w.close()
    handles = (_native.c_void_p * 1)(v.handle)
    blob, a, b, c, d = _native.pack_items([alpha], [ad])
    out = _native.ctypes.create_string_buffer(1)
    ok = _native.c_int(0)
    idx = (_native.c_uint32 * 1)(1)
    coeffs = b"".join(int(x).to_bytes(32, "little") for x in co)
    assert ctx.library.lib.dr_ring_verify_multi(ctx.handle, handles, 1, idx, 1, blob, a, b, c, d, proof, coeffs, 0, out, _native.ctypes.byref(ok)) == _native.DR_EINVAL
    for bad in (256, 1000, 1 << 17):
        assert refused(lambda: _native.NativeRingVerifier(ctx, root, g1_0, g2, domain_size=bad, omega=params.omega, seed=ps.accumulator_base,
                                                          blinding_base=ps.blinding_base, generator=bs.GENERATOR, suite_id=ps.suite_id, h2c_dst=ps.dst))
    assert multi([v], [], [], [], [], []) == ([], True)
    v.close()


def pool_matches_one_engine(api, engine, pool, items=None) -> None:
    """A RingVerifier over an EnginePool (one replica per device, contiguous shards) gives the verdicts of one engine."""
    items = items if items is not None else mixed_domain_items()
    roots = list(dict.fromkeys((r, p.domain_size, p.max_ring_size) for r, p, _, _, _ in items))
    params = [api.RingProofParams(domain_size=k[1], max_ring_size=k[2], test_vectors=True) for k in roots]
    index = [roots.index((r, p.domain_size, p.max_ring_size)) for r, p, _, _, _ in items]
    alphas, ads, proofs = [i[2] for i in items], [i[3] for i in items], [i[4] for i in items]
    ads_bad = list(ads)
    ads_bad[len(ads) // 2] += b"!"
    one = api.RingVerifier([api.RingRoot.decode(k[0], p) for k, p in zip(roots, params)], engine)
    many = api.RingVerifier([api.RingRoot.decode(k[0], p) for k, p in zip(roots, params)], pool)
    assert len(many.replicas) == len(pool)
    for d in (ads, ads_bad):
        want = one.verify_batch(proofs, alphas, d, index)
        assert many.verify_batch(proofs, alphas, d, index) == want
        assert want == [int(x == y) for x, y in zip(d, ads)]
        assert many.batch_verify(proofs, alphas, d, index) == one.batch_verify(proofs, alphas, d, index) == (d is ads)
    one.close()
    many.close()
