"""GPU run of the keyless, multi-ring verifier cases (tests/ring_verifier_cases.py) on cuda:0: the full sets, the ring-1023 reference
proofs, and 4096 proofs over eight rings of 1023 keys against 64 verifiers."""

import random

import pytest

from tests import ring_verifier_cases as cases
from tests.ring_fixtures import native_ring, native_srs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from dot_ring_b200 import _native

    c = _native.Context(0)
    assert c.library.is_cuda
    yield c
    c.close()


@pytest.fixture(scope="module")
def srs(ctx):
    s = native_srs(ctx, None, 10)
    yield s
    s.close()


@pytest.fixture(scope="module")
def api():
    import dot_ring_b200 as pkg

    return pkg


def test_keyless_reference_vectors(ctx):
    cases.keyless_reference_vectors(ctx)


def test_mixed_domains_with_ring1023(ctx):
    cases.mixed_domains(ctx, with_ring1023=True)


def test_same_as_keyed_path_full_sweep(ctx, srs):
    cases.same_as_keyed(ctx, srs, one_per_type=False)


def test_oracle_parity_across_rings(ctx):
    cases.oracle_parity_across_rings(ctx, cases.mixed_domain_items(with_ring1023=True))


def test_adversarial_roots(ctx):
    cases.adversarial_roots(ctx)


def test_abi_errors(ctx):
    from dot_ring_b200 import _native

    other = _native.Context(0)
    try:
        cases.errors_at_the_abi(ctx, other)
    finally:
        other.close()


def test_no_window_table(api):
    from dot_ring_b200 import engine as engine_mod

    eng = engine_mod.Engine(0)
    try:
        cases.no_window_table(api, eng)
    finally:
        eng.close()


def test_api_edges(api):
    from dot_ring_b200 import engine as engine_mod

    eng = engine_mod.Engine(0, window_bits=8, srs_points=1537)
    try:
        cases.api_edges(api, eng)
    finally:
        eng.close()


def test_4096_proofs_over_8_rings_64_verifiers(ctx, srs, api):
    """Proofs by the existing prover over eight rings of 1023 keys (512 per ring, every 37th item with a wrong ad), verified in one
    call against 64 verifiers (the eight rings at scattered indices, 56 decoys): per item equal to each ring's own
    dr_ring_verify_batch, aggregated through both routes; a RingVerifier over EnginePool([0, 0]) gives the same verdicts."""
    from dot_ring_b200 import engine as engine_mod
    from oracle import bandersnatch as bs
    from oracle import fr
    from oracle import ring_proof as rp
    from oracle import transcript as otr
    from tests.helpers import bench_ring_keys, le64, seed

    params = rp.Params.from_ring_size(1023)
    _, sk, base = bench_ring_keys(1023)

    rings, roots = [], []
    for r in range(8):
        keys = list(base)
        if r:
            keys[1000] = otr.secret_from_seed(bs.SHA512, seed("multi-ring-test", r))[0]
        rings.append(native_ring(srs, keys, params))
        roots.append(rings[-1].root())
    assert len(set(roots)) == 8
    rng = random.Random(1)
    per = 512
    alphas, ads, proofs, ring_of = [], [], [], []
    for r in range(8):
        al = [b"multi-%d-" % r + le64(j) for j in range(per)]
        ad = [b"multi-ad-%d-" % r + le64(j) for j in range(per)]
        pr, st = rings[r].prove_batch(al, ad, [sk] * per, [3] * per, zk_rows=[rng.randrange(fr.R) for _ in range(12 * per)])
        assert not any(st)
        alphas += al
        ads += [d + (b"!" if (r * per + j) % 37 == 0 else b"") for j, d in enumerate(ad)]
        proofs += pr
        ring_of += [r] * per
    n = len(proofs)
    # 64 verifiers: ring r at index 8 r + 5, decoys elsewhere (the other rings' roots and the small-ring / ark-vrf roots)
    decoys = [(i[0], i[1]) for i in cases.mixed_domain_items()]
    slots, verifiers = {}, []
    for k in range(64):
        if k % 8 == 5:
            slots[k // 8] = k
            verifiers.append(cases.make_verifier(ctx, roots[k // 8], params))
        elif k % 3 == 0:
            verifiers.append(cases.make_verifier(ctx, roots[(k + 3) % 8], params))
        else:
            root, p = decoys[k % len(decoys)]
            verifiers.append(cases.make_verifier(ctx, root, p))
    index = [slots[r] for r in ring_of]
    co = cases.independent(n, 60)
    want = []
    for r in range(8):
        lo, hi = r * per, (r + 1) * per
        want += rings[r].verify_batch(alphas[lo:hi], ads[lo:hi], proofs[lo:hi], co[2 * lo : 2 * hi])[0]
    assert want == [0 if i % 37 == 0 else 1 for i in range(n)]
    assert cases.multi(verifiers, index, alphas, ads, proofs, co) == (want, False)
    co = cases.adv.coeffs_random(n, 61)
    assert cases.both_routes(verifiers, index, alphas, ads, proofs, co) == (want, False)  # a wrong ad fails the Pedersen part
    honest = [i for i in range(n) if i % 37]
    sel = lambda xs: [xs[i] for i in honest]  # noqa: E731
    co = cases.adv.coeffs_random(len(honest), 62)
    assert cases.both_routes(verifiers, sel(index), sel(alphas), sel(ads), sel(proofs), co) == ([1] * len(honest), True)
    for v in verifiers:
        v.close()
    # the same batch through RingVerifier: one engine and a two-device pool
    rp_params = api.RingProofParams.from_ring_size(1023)
    root_objs = [api.RingRoot.decode(rt, rp_params) for rt in roots]
    eng = engine_mod.Engine(0, srs_points=1537)
    pool = engine_mod.EnginePool(devices=[0, 0], srs_points=1537)
    try:
        one = api.RingVerifier(root_objs, eng)
        many = api.RingVerifier(root_objs, pool)
        assert one.verify_batch(proofs, alphas, ads, ring_of) == want
        assert many.verify_batch(proofs, alphas, ads, ring_of) == want
        assert not many.batch_verify(proofs, alphas, ads, ring_of)
        assert many.batch_verify(sel(proofs), sel(alphas), sel(ads), sel(ring_of)) and one.batch_verify(sel(proofs), sel(alphas), sel(ads), sel(ring_of))
        assert eng._srs is None and all(e._srs is None for e in pool.engines)
        one.close()
        many.close()
    finally:
        eng.close()
        pool.close()
    for r in rings:
        r.close()


def test_pool_matches_one_engine(api):
    from dot_ring_b200 import engine as engine_mod

    eng = engine_mod.Engine(0, srs_points=1537)
    pool = engine_mod.EnginePool(devices=[0, 0], srs_points=1537)
    try:
        cases.pool_matches_one_engine(api, eng, pool, cases.mixed_domain_items(with_ring1023=True))
    finally:
        eng.close()
        pool.close()
