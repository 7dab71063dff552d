"""CPU run of the bare ring-proof cases (tests/ring_proof_prove_cases.py) through the test-only emulation build: SRS of 1537 points,
so every ring is on N = 512."""

import pytest

from dot_ring_b200 import _native
from dot_ring_b200 import engine as engine_mod
from tests import ring_proof_prove_cases as cases
from tests.host.emul import emulation_library
from tests.ring_fixtures import native_srs


@pytest.fixture(scope="module")
def ctx():
    c = _native.Context(0, emulation_library())
    yield c
    c.close()


@pytest.fixture(scope="module")
def srs(ctx):
    s = native_srs(ctx, 1537, 4)
    yield s
    s.close()


@pytest.fixture(scope="module")
def engine():
    lib = emulation_library()
    old = _native._default
    _native.set_default_library(lib)
    eng = engine_mod.Engine(0, window_bits=4, library=lib, srs_points=1537)
    engine_mod.set_default_engine(eng, 0)
    yield eng
    engine_mod.set_default_engine(None, 0)
    eng.close()
    _native.set_default_library(old)


@pytest.fixture(scope="module")
def api(engine):
    import dot_ring_b200 as pkg

    return pkg


def test_composition_with_pedersen_matches_ark_vectors(ctx, srs):
    cases.composition_ark_vectors(ctx, srs)


def test_custom_label_matches_oracle(ctx, srs):
    cases.custom_label(ctx, srs)


def test_round_trip_through_verifier(ctx, srs):
    cases.round_trip(ctx, srs)


def test_several_rings_on_every_route(ctx, srs):
    cases.several_rings(ctx, srs)


def test_errors(ctx, srs):
    other_srs = native_srs(ctx, 1537, 4)
    try:
        cases.errors(ctx, srs, other_srs)
    finally:
        other_srs.close()


def test_api_round_trip(api, engine):
    cases.api_round_trip(api, engine)


def test_pool_matches_one_engine(api, engine):
    pool = engine_mod.EnginePool(devices=[0, 0], window_bits=4, library=emulation_library(), srs_points=1537)
    try:
        cases.pool_matches_one_engine(api, engine, pool)
    finally:
        pool.close()
