"""GPU run of the multi-ring prover cases (tests/ring_prove_multi_cases.py) on cuda:0: N = 512 and N = 2048 rings in one call with the
reference's proofs byte-exact, and 4096 proofs over eight rings of 1023 keys, on one device and through a two-device EnginePool."""

import pytest

from tests import ring_prove_multi_cases as cases
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


def test_same_bytes_as_one_ring_at_a_time_on_every_route(ctx, srs):
    cases.same_bytes(ctx, srs, per_ring=3)


def test_mixed_domains_byte_exact(ctx, srs):
    """N = 512 and N = 2048 rings in one call, with the six ring-1023 reference proofs (4 zeroed, 2 blinded rows) and the N = 2048
    max_ring_size 6 proof of small_ring_reference.json, on every route."""
    cases.same_bytes(ctx, srs, per_ring=2, with_2048=True)


def test_status_per_item(ctx, srs):
    cases.status_per_item(ctx, srs)


def test_api_round_trip_and_key_errors(api):
    from dot_ring_b200 import engine as engine_mod

    eng = engine_mod.Engine(0, window_bits=8, srs_points=1537)
    try:
        cases.api_round_trip(api, eng)
    finally:
        eng.close()


def test_errors(ctx, srs):
    from dot_ring_b200 import _native

    other_srs = native_srs(ctx, 1537, 8)
    other_ctx = _native.Context(0)
    other_ctx_srs = native_srs(other_ctx, 1537, 8)
    try:
        cases.errors(ctx, srs, other_srs, other_ctx, other_ctx_srs)
    finally:
        other_srs.close()
        other_ctx_srs.close()
        other_ctx.close()


def test_pool_matches_one_engine(api):
    from dot_ring_b200 import engine as engine_mod

    eng = engine_mod.Engine(0, window_bits=8)
    pool = engine_mod.EnginePool(devices=[0, 0], window_bits=8)
    try:
        cases.pool_matches_one_engine(api, eng, pool, with_2048=True)
    finally:
        eng.close()
        pool.close()


def test_4096_proofs_over_8_rings(ctx, srs, api):
    """4096 proofs over eight distinct rings of 1023 keys, interleaved: every proof equals its ring's own dr_ring_prove_batch, in one
    dr_ring_prove_multi call on one device and through RingVRF.prove_multi over a two-device EnginePool."""
    from dot_ring_b200 import engine as engine_mod

    keys, params, items = cases.eight_rings_1023(srs)
    natives = [native_ring(srs, k, params) for k in keys]
    assert len({r.root() for r in natives}) == 8
    want = cases.one_ring_at_a_time(natives, items)
    proofs, status = cases.prove_multi(natives, items)
    assert status == [0] * len(items)
    assert proofs == want
    for r in natives:
        r.close()
    cls = api.RingVRF[api.Bandersnatch]
    pool = engine_mod.EnginePool(devices=[0, 0], window_bits=10)
    try:
        rp_params = api.RingProofParams.from_ring_size(1023)
        rings = [api.Ring(k, rp_params, pool) for k in keys]
        got = cls.prove_multi([it[1] for it in items], [it[2] for it in items], [it[3] for it in items], [it[4] for it in items], rings, [it[0] for it in items],
                              zk_rows=cases.zk_of(items), as_bytes=True)
        assert got == want
        for r in rings:
            r.native.close()
    finally:
        pool.close()
