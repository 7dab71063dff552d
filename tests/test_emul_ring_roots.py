"""CPU run of the ring-root cases (tests/ring_root_cases.py) through the test-only emulation build, at N = 512 (the N = 2048
reference ring of small_ring_reference.json included)."""

import pytest

from dot_ring_b200 import _native
from dot_ring_b200 import engine as engine_mod
from oracle import ring_proof as rp
from tests import ring_root_cases as cases
from tests.host.emul import emulation_library
from tests.ring_fixtures import native_srs
from tests.verify_cases import SUITES


@pytest.fixture(scope="module")
def ctx():
    c = _native.Context(0, emulation_library())
    yield c
    c.close()


@pytest.fixture(scope="module")
def srs_for(ctx):
    """N -> the first N bundled SRS points with the root table (built once per N)."""
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


def test_reference_pins(srs_for):
    cases.reference_pins(srs_for)


@pytest.mark.parametrize("suite", [s for s, _ in SUITES], ids=[p for _, p in SUITES])
def test_same_as_ring_create(ctx, srs_for, ring_srs, suite):
    cases.same_as_ring_create(ctx, srs_for(512), ring_srs, rp.Params(suite=suite))


def test_batching(ctx, srs_for, ring_srs):
    cases.batching(ctx, srs_for(512), ring_srs, rp.Params())


def test_update_walk(ctx, srs_for, ring_srs):
    cases.update_walk(ctx, srs_for(512), ring_srs, rp.Params(), steps=20, seed=1)


def test_abi_errors(ctx, srs_for):
    other = _native.Context(0, emulation_library())
    try:
        cases.abi_errors(ctx, other, srs_for(512), rp.Params(test_vectors=True))
    finally:
        other.close()


def test_api_errors(api, engine):
    cases.api_errors(api, engine)


def test_api_semantics(api, engine):
    cases.api_semantics(api, engine)


def test_no_window_table(api):
    eng = engine_mod.Engine(0, window_bits=4, library=emulation_library(), srs_points=1537)
    try:
        cases.no_window_table(api, eng)
    finally:
        eng.close()


def test_pool_matches_one_engine(api, engine):
    pool = engine_mod.EnginePool(devices=[0, 0], window_bits=4, library=emulation_library(), srs_points=1537)
    try:
        cases.pool_matches_one_engine(api, engine, pool)
    finally:
        pool.close()
