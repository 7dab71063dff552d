"""GPU run of the adversarial parity cases (tests/adversarial_cases.py) on cuda:0: the full set, ring 8 and ring 1023."""

import pytest

from tests import adversarial_cases as cases
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


def test_subgroup_test_matches_point_order():
    cases.subgroup_test_matches_order()


def test_g1_msm_off_subgroup(ctx):
    cases.msm_off_subgroup(ctx, [1, 2, 33, 2048])


def test_g1_msm_off_subgroup_through_engine_pool():
    from dot_ring_b200 import engine as engine_mod

    pool = engine_mod.EnginePool(devices=[0, 0], window_bits=4, srs_points=1537)
    try:
        cases.msm_off_subgroup(pool.engines[0].ctx, [33, 2048], pool=pool)
    finally:
        pool.close()


def test_pairing_off_subgroup(ctx):
    cases.pairing_off_subgroup(ctx)


def test_vrf_tamper_sweep_both_kernels(ctx):
    cases.vrf_tamper_sweep_both_kernels(ctx)


def test_ring8_tamper_sweep(srs):
    cases.ring_tamper_sweep(srs)


def test_ring1023_tamper_sweep(srs):
    cases.ring1023_tamper_sweep(srs)


def test_coefficient_exact_openings(srs):
    cases.coefficient_exact_openings(srs)


def test_batch_binding_and_pool(srs):
    from dot_ring_b200 import engine as engine_mod

    eng = engine_mod.Engine(0, window_bits=4, srs_points=1537)
    engine_mod.set_default_engine(eng, 0)
    pool = engine_mod.EnginePool(devices=[0, 0], window_bits=4, srs_points=1537)
    try:
        import dot_ring_b200 as api

        keys = [pk for pk, _ in cases._signers()]
        params = api.RingProofParams()
        ring_pool = api.Ring(keys, params, pool)
        root = api.RingRoot.from_ring(ring_pool, params)
        cls = api.RingVRF[api.Bandersnatch]
        keys, alphas, ads, proofs = cases.batch_binding(srs, n=7, pool_ring=lambda a, d, p, co: cls.verify_batch(p, a, d, ring_pool, root))
        cases.wrong_ring_through_api(api, keys, alphas, ads, proofs)
    finally:
        pool.close()
        engine_mod.set_default_engine(None, 0)
        eng.close()
