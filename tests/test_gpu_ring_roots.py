"""GPU run of the ring-root cases (tests/ring_root_cases.py) on cuda:0: N = 512, 2048 and 4096 against dr_ring_create, N = 65536 over
a synthetic SRS, the ring-1023 reference root, a longer update sequence, and proofs of RingVRF.prove_batch accepted against roots
from keys."""

import pytest

from oracle import ring_proof as rp
from tests import ring_root_cases as cases
from tests.ring_fixtures import native_srs
from tests.verify_cases import SUITES

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from dot_ring_b200 import _native

    c = _native.Context(0)
    assert c.library.is_cuda
    yield c
    c.close()


@pytest.fixture(scope="module")
def srs_for(ctx):
    made = {}

    def get(n):
        if n not in made:
            made[n] = cases.root_srs(ctx, n)
        return made[n]

    yield get
    for s in made.values():
        s.close()


@pytest.fixture(scope="module")
def ring_srs(ctx):
    s = native_srs(ctx, None, 10)  # the bundled 6145 points = 3N + 1 at N = 2048
    yield s
    s.close()


@pytest.fixture(scope="module")
def api():
    import dot_ring_b200 as pkg

    return pkg


@pytest.fixture(scope="module")
def engine():
    from dot_ring_b200 import engine as engine_mod

    eng = engine_mod.Engine(0, window_bits=8, srs_points=1537)
    yield eng
    eng.close()


def full_params(domain: int, suite) -> rp.Params:
    return rp.Params(domain_size=domain, max_ring_size=domain - rp.SCALAR_BITS - 4, suite=suite, max_domain_size=max(domain, 4096))


def test_reference_pins(srs_for):
    cases.reference_pins(srs_for)


def test_ring1023_reference_root(srs_for):
    cases.ring1023_pin(srs_for(2048))


@pytest.mark.parametrize("domain", [512, 2048])
@pytest.mark.parametrize("suite", [s for s, _ in SUITES], ids=[p for _, p in SUITES])
def test_same_as_ring_create(ctx, srs_for, ring_srs, suite, domain):
    cases.same_as_ring_create(ctx, srs_for(domain), ring_srs, full_params(domain, suite), seed=domain)


@pytest.mark.parametrize("suite", [s for s, _ in SUITES], ids=[p for _, p in SUITES])
def test_same_as_ring_create_4096(ctx, suite):
    """N = 4096 needs 12289 points for dr_ring_create: both sides run over one synthetic SRS."""
    ring_srs = cases.synthetic_ring_srs(ctx, 3 * 4096 + 1, 8)
    srs = cases.root_srs(ctx, 4096, cases.synthetic_g1(ctx, 4096))
    try:
        cases.same_as_ring_create(ctx, srs, ring_srs, full_params(4096, suite), seed=4096)
    finally:
        srs.close()
        ring_srs.close()


def test_large_domain_65536(ctx):
    cases.large_domain(ctx, n_keys=5000, domain=65536, ring_window_bits=4)


def test_batching(ctx, srs_for, ring_srs):
    cases.batching(ctx, srs_for(2048), ring_srs, full_params(2048, SUITES[0][0]), counts=(1023, 0, 1, 1791, 0, 5, 200, 17))


def test_batching_over_passes(ctx, srs_for):
    """1030 rings in one call run as two passes of at most 1024 rings (C_s committed in the first only): every root equals its own
    single-ring call."""
    params = rp.Params()
    keys = cases.fresh_keys(ctx, 16, 200)
    sets = [keys[i % 7 : i % 7 + i % 5] for i in range(1030)]
    srs = srs_for(512)
    got = cases.roots(srs, params, sets)
    singles = {}
    for keys_i, root in zip(sets, got):
        key = tuple(keys_i)
        if key not in singles:
            singles[key] = cases.roots(srs, params, [keys_i])[0]
        assert root == singles[key]
    assert len(singles) == 29  # seven offsets x four lengths, and the empty ring


def test_update_walk(ctx, srs_for, ring_srs):
    cases.update_walk(ctx, srs_for(2048), ring_srs, full_params(2048, SUITES[0][0]), steps=120, seed=2)


def test_update_walk_small_ring(ctx, srs_for, ring_srs):
    """max_ring_size 6 at N = 2048 (as the reference's small rings): appends stop at the last key row."""
    cases.update_walk(ctx, srs_for(2048), ring_srs, rp.Params(domain_size=2048, max_ring_size=6), steps=40, seed=3)


def test_abi_errors(ctx, srs_for):
    from dot_ring_b200 import _native

    other = _native.Context(0)
    try:
        cases.abi_errors(ctx, other, srs_for(512), rp.Params(test_vectors=True))
    finally:
        other.close()


def test_api_errors(api, engine):
    cases.api_errors(api, engine)


def test_api_semantics(api, engine):
    cases.api_semantics(api, engine)


def test_no_window_table(api):
    from dot_ring_b200 import engine as engine_mod

    eng = engine_mod.Engine(0)
    try:
        cases.no_window_table(api, eng)
    finally:
        eng.close()


def test_pool_matches_one_engine(api, engine):
    from dot_ring_b200 import engine as engine_mod

    pool = engine_mod.EnginePool(devices=[0, 0], srs_points=1537)
    try:
        cases.pool_matches_one_engine(api, engine, pool)
    finally:
        pool.close()


def test_prove_batch_round_trip(api):
    """Proofs of RingVRF.prove_batch over Ring(keys) verify against RingVerifier([RingRoot.from_keys(keys, params)]) on an engine that
    never builds the prover's table, per item and aggregated; a proof under a wrong ad does not."""
    from dot_ring_b200 import engine as engine_mod
    from tests.helpers import bench_ring_keys, le64

    pk, sk, keys = bench_ring_keys(1023)
    params = api.RingProofParams.from_ring_size(1023)
    prover = engine_mod.Engine(0, window_bits=10)
    verifier_engine = engine_mod.Engine(0)
    try:
        ring = api.Ring(keys, params, prover)
        n = 64
        alphas, ads = [b"round-trip-" + le64(j) for j in range(n)], [b"ad-" + le64(j) for j in range(n)]
        proofs = api.RingVRF[api.Bandersnatch].prove_batch(alphas, ads, sk, pk, ring, as_bytes=True)
        root = api.RingRoot.from_keys(keys, params, verifier_engine)
        assert root.fixed_commitments() == api.RingRoot.from_ring(ring).fixed_commitments()
        verifier = api.RingVerifier([root], verifier_engine)
        assert verifier.verify_batch(proofs, alphas, ads) == [1] * n
        assert verifier.batch_verify(proofs, alphas, ads)
        bad = list(ads)
        bad[7] += b"!"
        assert verifier.verify_batch(proofs, alphas, bad) == [1] * 7 + [0] + [1] * (n - 8)
        assert not verifier.batch_verify(proofs, alphas, bad)
        verifier.close()
        assert verifier_engine._srs is None
    finally:
        prover.close()
        verifier_engine.close()
