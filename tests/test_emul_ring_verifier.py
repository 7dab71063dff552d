"""CPU run of the keyless, multi-ring verifier cases (tests/ring_verifier_cases.py) through the test-only emulation build."""

import pytest

from dot_ring_b200 import _native
from dot_ring_b200 import engine as engine_mod
from tests import ring_verifier_cases as cases
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


def test_keyless_reference_vectors(ctx):
    cases.keyless_reference_vectors(ctx)


def test_mixed_domains(ctx):
    cases.mixed_domains(ctx)


def test_same_as_keyed_path(ctx, srs):
    cases.same_as_keyed(ctx, srs, one_per_type=True, fold_sample=3)


def test_oracle_parity_across_rings(ctx):
    cases.oracle_parity_across_rings(ctx)


def test_adversarial_roots(ctx):
    cases.adversarial_roots(ctx)


def test_abi_errors(ctx):
    other = _native.Context(0, emulation_library())
    try:
        cases.errors_at_the_abi(ctx, other)
    finally:
        other.close()


def test_no_window_table(api):
    eng = engine_mod.Engine(0, window_bits=4, library=emulation_library(), srs_points=1537)
    try:
        cases.no_window_table(api, eng)
    finally:
        eng.close()


def test_api_edges(api, engine):
    cases.api_edges(api, engine)


def test_pool_matches_one_engine(api, engine):
    pool = engine_mod.EnginePool(devices=[0, 0], window_bits=4, library=emulation_library(), srs_points=1537)
    try:
        cases.pool_matches_one_engine(api, engine, pool)
    finally:
        pool.close()
