"""CPU checks of the product's __host__ __device__ math headers (host-compiled into a test-only
library) against the oracle: Fq / Fr / Fn arithmetic, G1 group law + zcash codecs, Bandersnatch
decode / scalar-mul / Elligator2, SHA-512 and SHAKE128.  Mirrors the reference's
tests/test_curve_ops/test_native_field.py (random add/sub/mul vs Python ints)."""

import ctypes
import hashlib
import random
import subprocess
from pathlib import Path

import pytest

from oracle import bandersnatch as bs
from oracle import bls12_381 as bls
from oracle import fr
from tests.helpers import load

HERE = Path(__file__).resolve().parent / "host"


@pytest.fixture(scope="module")
def lib():
    so = HERE / "libdr_hosttest.so"
    src = HERE / "hosttest.cpp"
    hdrs = list((HERE.parents[1] / "dot_ring_b200" / "csrc").glob("*.cuh")) + list((HERE.parents[1] / "dot_ring_b200" / "csrc" / "gen").glob("*"))
    if not so.exists() or so.stat().st_mtime < max(p.stat().st_mtime for p in [src, *hdrs]):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-DDR_HOST_EMULATION", "-shared", "-fPIC", "-o", str(so), str(src)])
    return ctypes.CDLL(str(so))


def _buf(n):
    return ctypes.create_string_buffer(n)


def test_fq_ops(lib):
    rng = random.Random(1)
    P = bls.P
    vals = [0, 1, 2, P - 1, P - 2, (1 << 380), P >> 1] + [rng.randrange(P) for _ in range(100)]
    for _ in range(200):
        a, b = rng.choice(vals), rng.choice(vals)
        for op, want in ((0, a * b % P), (1, (a + b) % P), (2, (a - b) % P), (5, a * a % P)):
            out = _buf(48)
            lib.ht_fq_op(op, a.to_bytes(48, "big"), b.to_bytes(48, "big"), out)
            assert int.from_bytes(out.raw, "big") == want, (op, a, b)
    for a in vals[:20]:
        out = _buf(48)
        lib.ht_fq_op(3, a.to_bytes(48, "big"), bytes(48), out)
        assert int.from_bytes(out.raw, "big") == (pow(a, -1, P) if a else 0)
        sq = a * a % P
        ok = lib.ht_fq_op(4, sq.to_bytes(48, "big"), bytes(48), out)
        assert ok and int.from_bytes(out.raw, "big") in (a % P, (-a) % P)
    assert not lib.ht_fq_op(4, (2).to_bytes(48, "big"), bytes(48), _buf(48)) or pow(2, (P - 1) // 2, P) == 1


def test_fr_ops(lib):
    rng = random.Random(2)
    P = bs.P
    vals = [0, 1, 2, P - 1, P - 2, 5, P >> 1] + [rng.randrange(P) for _ in range(100)]
    for _ in range(200):
        a, b = rng.choice(vals), rng.choice(vals)
        for op, want in ((0, a * b % P), (1, (a + b) % P), (2, (a - b) % P), (5, a * a % P)):
            out = _buf(32)
            lib.ht_fr_op(op, a.to_bytes(32, "little"), b.to_bytes(32, "little"), out)
            assert int.from_bytes(out.raw, "little") == want, (op, a, b)
    for a in vals[:40]:
        out = _buf(32)
        lib.ht_fr_op(3, a.to_bytes(32, "little"), bytes(32), out)
        assert int.from_bytes(out.raw, "little") == (pow(a, -1, P) if a else 0)
        is_sq = lib.ht_fr_op(6, a.to_bytes(32, "little"), bytes(32), out)
        assert bool(is_sq) == bs.fr_is_square(a)
        ok = lib.ht_fr_op(4, a.to_bytes(32, "little"), bytes(32), out)
        assert bool(ok) == bs.fr_is_square(a)
        if ok:
            assert pow(int.from_bytes(out.raw, "little"), 2, P) == a


def test_fn_reduction_and_muladd(lib):
    rng = random.Random(3)
    for n in (16, 32, 48, 64):
        for _ in range(20):
            data = bytes(rng.randrange(256) for _ in range(n))
            out = _buf(32)
            lib.ht_fn_from_bytes_mod(data, n, out)
            assert int.from_bytes(out.raw, "little") == int.from_bytes(data, "little") % bs.N
    out = _buf(32)
    lib.ht_fn_from_bytes_mod(b"\xff" * 64, 64, out)
    assert int.from_bytes(out.raw, "little") == (2**512 - 1) % bs.N
    for _ in range(20):
        k, c, x = (rng.randrange(bs.N) for _ in range(3))
        lib.ht_fn_muladd(k.to_bytes(32, "little"), c.to_bytes(32, "little"), x.to_bytes(32, "little"), out)
        assert int.from_bytes(out.raw, "little") == (k + c * x) % bs.N


def test_g1_group_law_and_codecs(lib):
    rng = random.Random(4)
    g = (bls.G1_GEN[0], bls.G1_GEN[1], 1)
    pts = [bls.g1_mul(g, rng.randrange(bls.R)) for _ in range(6)]
    for p in pts:
        ser, comp = bls.g1_serialize(p), bls.g1_compress(p)
        out96, out48 = _buf(96), _buf(48)
        assert lib.ht_g1_decode(comp, 48, out96) and out96.raw == ser
        assert lib.ht_g1_decode(ser, 96, out96) and out96.raw == ser
        lib.ht_g1_compress(ser, out48)
        assert out48.raw == comp
        k = rng.randrange(bls.R)
        want = bls.g1_serialize(bls.g1_mul(p, k))
        lib.ht_g1_mul(ser, k.to_bytes(32, "little"), out96)
        assert out96.raw == want
        lib.ht_g1_mul_mixed(ser, k.to_bytes(32, "little"), out96)
        assert out96.raw == want
    a, b = pts[0], pts[1]
    inf = bls.g1_serialize(None)
    for x, y in ((a, b), (a, a), (a, bls.g1_neg(a)), (a, None), (None, a), (None, None)):
        for mode in (0, 1):
            out96 = _buf(96)
            lib.ht_g1_add(bls.g1_serialize(x), bls.g1_serialize(y), mode, out96)
            assert out96.raw == bls.g1_serialize(bls.g1_add(x, y)), (mode,)
    assert bls.g1_serialize(None) == inf
    # malformed encodings are rejected (blst raises -> ValueError in the reference)
    assert not lib.ht_g1_decode(b"\xff" * 48, 48, _buf(96))
    assert not lib.ht_g1_decode(bytes(48), 48, _buf(96))
    bad = bytearray(bls.g1_serialize(a))
    bad[95] ^= 1
    assert not lib.ht_g1_decode(bytes(bad), 96, _buf(96))
    out96 = _buf(96)
    assert lib.ht_g1_decode(bytes([0xC0]) + bytes(47), 48, out96) and out96.raw == inf


def test_g1_subgroup_membership(lib):
    """msm.cuh g1_in_subgroup (the verifier's switch between the GLV split and a full multiplication) against [r]P == O."""
    from tests.adversarial_cases import in_g1, membership_points

    lib.ht_g1_in_subgroup.argtypes = [ctypes.c_char_p]
    for pt in membership_points(6):
        assert lib.ht_g1_in_subgroup(bls.g1_serialize(pt)) == int(in_g1(pt)), bls.g1_to_affine(pt)


def test_g1_full_multiplication_outside_the_subgroup(lib):
    """g1_mul_limbs on small-order points and points with a small-order component: multiples inside its window table reach
    infinity (3T, 6T, ... for a point T of order 3), and the product must still be the integer multiple k * P."""
    from tests.adversarial_cases import membership_points

    rng = random.Random(12)
    for pt in membership_points(4):
        for k in (1, 2, 3, 6, 11, 15, 0x1234567, bls.R - 1, rng.randrange(bls.R)):
            out = _buf(96)
            lib.ht_g1_mul_limbs(bls.g1_serialize(pt), k.to_bytes(32, "little"), out)
            assert out.raw == bls.g1_serialize(bls.g1_mul_raw(pt, k)), (bls.g1_to_affine(pt), k)


def test_batched_affine_round_exceptional_cases(lib):
    """msm.cuh affine_round: generic pairs share one inversion with P + P (denominator 2y), P - P and infinity operands."""
    rng = random.Random(9)
    g = (bls.G1_GEN[0], bls.G1_GEN[1], 1)
    p = [bls.g1_mul(g, rng.randrange(1, bls.R)) for _ in range(8)]
    pairs = [(p[0], p[1]), (p[2], p[2]), (p[3], bls.g1_neg(p[3])), (None, p[4]), (p[5], None), (None, None), (p[6], p[7]), (p[1], p[0]), (p[7], p[7])]
    data = b"".join(bls.g1_serialize(x) + bls.g1_serialize(y) for x, y in pairs)
    out = _buf(96 * len(pairs))
    lib.ht_affine_round(data, 2 * len(pairs), out)
    for i, (x, y) in enumerate(pairs):
        assert out.raw[96 * i : 96 * i + 96] == bls.g1_serialize(bls.g1_add(x, y)), i


def test_modular_inverses_and_legendre_symbol(lib):
    """fp.cuh inv() (Bernstein-Yang division steps), inv_kaliski() and Fermat's x^(p-2) against Python's pow; legendre() against
    Euler's criterion."""
    rng = random.Random(12)
    for field, mod, size, order in ((0, bls.P, 48, "big"), (1, fr.R, 32, "little")):
        edge = [0, 1, 2, 3, 4, mod - 1, mod - 2, (mod - 1) // 2, (mod + 1) // 2, 1 << 200, (1 << 32) - 1, 1 << 32]
        for v in edge + [rng.randrange(mod) for _ in range(300)] + [rng.randrange(1 << k) for k in range(1, 64, 3)] + [mod - rng.randrange(1, 1 << 40) for _ in range(20)]:
            out, out2, out3 = _buf(size), _buf(size), _buf(size)
            sym = lib.ht_inv_and_legendre(field, v.to_bytes(size, order), out, out2, out3)
            want = pow(v, -1, mod) if v else 0
            assert int.from_bytes(out.raw, order) == want == int.from_bytes(out2.raw, order) == int.from_bytes(out3.raw, order), (field, v)
            euler = 0 if v == 0 else (1 if pow(v, (mod - 1) // 2, mod) == 1 else -1)
            assert sym == euler, (field, v)


def test_subgroup_test_by_two_descent(lib):
    """te.cuh te_in_prime_subgroup: two Legendre symbols must agree with [n]P == O on points of all four cosets of E / 2E,
    on the identity and on the 2-torsion point (0, -1)."""
    rng = random.Random(13)
    seen = {1: 0, 0: 0}
    t2 = (0, bs.P - 1)
    for _ in range(60):
        while True:
            y = rng.randrange(bs.P)
            den = (bs.A - bs.D * y * y) % bs.P
            x = bs.fr_sqrt((1 - y * y) * pow(den, -1, bs.P) % bs.P) if den else None
            if x is not None:
                break
        for pt in ((x, y), (bs.P - x, y)):
            got = lib.ht_te_subgroup(pt[0].to_bytes(32, "little") + pt[1].to_bytes(32, "little"))
            assert got in (0, 3), (pt, got)
            seen[got & 1] += 1
            if got == 3:  # P in the subgroup: P + (0, -1) = (-x, -y) is not
                q = ((-pt[0]) % bs.P, (-pt[1]) % bs.P)
                assert lib.ht_te_subgroup(q[0].to_bytes(32, "little") + q[1].to_bytes(32, "little")) == 0
    assert seen[1] > 5 and seen[0] > 20
    g = bs.mul(bs.GENERATOR, 12345)
    enc = lambda p: p[0].to_bytes(32, "little") + p[1].to_bytes(32, "little")  # noqa: E731
    assert lib.ht_te_subgroup(enc(g)) == 3 and lib.ht_te_subgroup(enc(bs.IDENTITY)) == 3 and lib.ht_te_subgroup(enc(t2)) == 0


def test_glv_split_and_multiplication(lib):
    """te.cuh te_glv_split / te_endomorphism / te_mul_glv: k = k1 + k2 lambda (mod n) with 128-bit halves, and the joint
    multiplication equals the plain one (oracle) -- incl. scalars 0, 1, n - 1 and the reference's golden scalar multiplications."""
    lam = 0x13B4F3DC4A39A493EDF849562B38C72BCFC49DB970A5056ED13D21408783DF05
    rng = random.Random(14)
    g = load("bandersnatch_reference.json")
    cases = [(bytes.fromhex(e["base"]), int(e["k"], 16), bytes.fromhex(e["out"])) for e in g["scalar_mul"]]
    base = bs.mul(bs.GENERATOR, 777)
    for k in [0, 1, 2, bs.N - 1, bs.N - 2, bs.N // 2, (1 << 252) - 1] + [rng.randrange(bs.N) for _ in range(40)]:
        cases.append((bs.point_to_string(base), k, bs.point_to_string(bs.mul(base, k))))
    for enc, k, want in cases:
        out, split = _buf(32), _buf(32)
        signs = lib.ht_te_mul_glv(enc, (k % bs.N).to_bytes(32, "little"), out, split)
        assert signs >= 0, signs
        k1 = int.from_bytes(split.raw[:16], "little") * (-1 if signs & 1 else 1)
        k2 = int.from_bytes(split.raw[16:], "little") * (-1 if signs & 2 else 1)
        assert (k1 + k2 * lam - k) % bs.N == 0 and abs(k1) < 1 << 127 and abs(k2) < 1 << 127
        assert out.raw == want, hex(k)


def test_bandersnatch_against_reference_goldens(lib):
    g = load("bandersnatch_reference.json")
    for e in g["dec_point"]:
        xy = _buf(64)
        ok = lib.ht_te_decode(bytes.fromhex(e["raw"]), 1, xy)
        assert bool(ok) == e["ok"]
        if ok:
            assert int.from_bytes(xy.raw[:32], "little") == int(e["x"], 16)
            assert int.from_bytes(xy.raw[32:], "little") == int(e["y"], 16)
    for e in g["scalar_mul"]:
        out = _buf(32)
        lib.ht_te_mul(bytes.fromhex(e["base"]), int(e["k"], 16).to_bytes(32, "little"), out)
        assert out.raw.hex() == e["out"]
    for e in g["encode_to_curve"]:
        u = bs.expand_message_xmd_sha512(bytes.fromhex(e["alpha"]), bs.SHA512.dst, 96)
        out = _buf(32)
        lib.ht_te_ell2(u[:48], u[48:], out)
        assert out.raw.hex() == e["point"]
    rng = random.Random(5)
    pts = [bs.mul(bs.GENERATOR, rng.randrange(bs.N)) for _ in range(3)]
    ks = [rng.randrange(bs.N) for _ in range(3)]
    for n in (1, 2, 3):
        out = _buf(32)
        lib.ht_te_msm(b"".join(bs.point_to_string(p) for p in pts[:n]), b"".join(k.to_bytes(32, "little") for k in ks[:n]), n, out)
        assert out.raw == bs.point_to_string(bs.msm(pts[:n], ks[:n]))
    # a point of small order / outside the subgroup is rejected by the checked decode
    assert not lib.ht_te_decode(bs.point_to_string((0, bs.P - 1)), 1, _buf(64))
    assert not lib.ht_te_decode(bs.point_to_string(bs.IDENTITY), 1, _buf(64))


def test_hashes(lib):
    rng = random.Random(6)
    for n in (0, 1, 55, 111, 112, 113, 127, 128, 129, 167, 168, 169, 335, 336, 1000, 2200):
        msg = bytes(rng.randrange(256) for _ in range(n))
        out = _buf(64)
        lib.ht_sha512(msg, n, out)
        assert out.raw == hashlib.sha512(msg).digest()
        for outlen in (48, 200):
            o2 = _buf(outlen)
            lib.ht_shake128(msg, n, o2, outlen)
            assert o2.raw == hashlib.shake_128(msg).digest(outlen)
