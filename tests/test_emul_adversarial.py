"""CPU run of the adversarial parity cases (tests/adversarial_cases.py) through the test-only emulation build: a reduced set."""

import pytest

from dot_ring_b200 import _native
from dot_ring_b200 import engine as engine_mod
from tests import adversarial_cases as cases
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
def api():
    lib = emulation_library()
    old = _native._default
    _native.set_default_library(lib)
    eng = engine_mod.Engine(0, window_bits=4, library=lib, srs_points=1537)
    engine_mod.set_default_engine(eng, 0)
    import dot_ring_b200 as pkg

    yield pkg
    engine_mod.set_default_engine(None, 0)
    eng.close()
    _native.set_default_library(old)


def test_subgroup_test_matches_point_order():
    cases.subgroup_test_matches_order(n_random=4)


def test_g1_msm_off_subgroup(ctx):
    cases.msm_off_subgroup(ctx, [1, 2, 33])


def test_pairing_off_subgroup(ctx):
    cases.pairing_off_subgroup(ctx)


def test_vrf_tamper_sweep_both_kernels(ctx):
    cases.vrf_tamper_sweep_both_kernels(ctx, cases.SUITES[:1])


def test_ring_tamper_sweep(srs):
    cases.ring_tamper_sweep(srs, full_sha=True, aggregate_sample=3)


def test_coefficient_exact_openings(srs):
    cases.coefficient_exact_openings(srs)


def test_batch_binding_and_pool(srs, api):
    lib = emulation_library()
    pool = engine_mod.EnginePool(devices=[0, 0], window_bits=4, library=lib, srs_points=1537)
    try:
        keys = [pk for pk, _ in cases._signers()]
        params = api.RingProofParams()
        ring_pool = api.Ring(keys, params, pool)
        root = api.RingRoot.from_ring(ring_pool, params)
        cls = api.RingVRF[api.Bandersnatch]
        keys, alphas, ads, proofs = cases.batch_binding(srs, n=5, pool_ring=lambda a, d, p, co: cls.verify_batch(p, a, d, ring_pool, root))
        cases.wrong_ring_through_api(api, keys, alphas, ads, proofs)
    finally:
        pool.close()
