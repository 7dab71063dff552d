"""GPU run of the bare ring-proof cases (tests/ring_proof_prove_cases.py) on cuda:0: the ark-vrf and ring-1023 reference proofs through
the Pedersen prover's blinding factors, another label at N = 2048, rings of N = 512 and 2048 in one call, 4096 proofs over eight rings of
1023 keys, and a two-device EnginePool."""

import pytest

from tests import ring_proof_prove_cases as cases
from tests.ring_fixtures import native_srs

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


def test_composition_with_pedersen_matches_ark_vectors(ctx, srs):
    cases.composition_ark_vectors(ctx, srs)


def test_composition_with_pedersen_matches_ring1023_reference(ctx, srs):
    cases.composition_ring1023(ctx, srs)


def test_custom_label_matches_oracle(ctx, srs):
    cases.custom_label(ctx, srs)


def test_custom_label_matches_oracle_2048(ctx, srs):
    cases.custom_label(ctx, srs, domain_size=2048)


def test_round_trip_through_verifier(ctx, srs):
    cases.round_trip(ctx, srs)


def test_several_rings_on_every_route(ctx, srs):
    cases.several_rings(ctx, srs, with_2048=True)


def test_errors(ctx, srs):
    other_srs = native_srs(ctx, 1537, 8)
    try:
        cases.errors(ctx, srs, other_srs)
    finally:
        other_srs.close()


def test_api_round_trip(api):
    from dot_ring_b200 import engine as engine_mod

    eng = engine_mod.Engine(0, window_bits=8, srs_points=1537)
    try:
        cases.api_round_trip(api, eng)
    finally:
        eng.close()


def test_pool_matches_one_engine(api):
    from dot_ring_b200 import engine as engine_mod

    eng = engine_mod.Engine(0, window_bits=8)
    pool = engine_mod.EnginePool(devices=[0, 0], window_bits=8)
    try:
        cases.pool_matches_one_engine(api, eng, pool, with_2048=True)
    finally:
        eng.close()
        pool.close()


def test_4096_proofs_over_8_rings(ctx, srs):
    cases.full_size_4096(ctx, srs)
