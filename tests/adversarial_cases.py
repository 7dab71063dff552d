"""Adversarial-input parity cases shared by the CPU (emulation build) and GPU (CUDA build) suites.

Every device verdict here is compared with the CPU oracle's verdict on the same bytes and the same batching coefficients
(2 = the reference's decode raises ValueError, else int(verify)); no expectation is hard-coded.  The inputs are what a
hostile prover or caller controls: every field of a proof replaced by malformed, non-canonical, small-order and
off-subgroup values, proofs recombined across a batch, openings forged for one exact pair of coefficients, and G1
points on the curve but outside G1 (decoding does not check the subgroup, as in blst's P1_Affine(bytes)).

Not covered: MSM scalars >= r on points outside G1.  The device reduces every scalar mod r first; on such points k * P and
(k mod r) * P differ, and which of the two blst is handed by the reference is not settled here."""

from __future__ import annotations

import random
from functools import lru_cache

from oracle import bandersnatch as bs
from oracle import bls12_381 as bls
from oracle import ring_proof as rp
from oracle import transcript as tr
from oracle import vrf as ovrf
from tests.helpers import hx, load, ring_proof_bytes, seed, split_keys
from tests.ring_fixtures import native_ring
from tests.verify_cases import SUITES, suite_struct

R = bls.R
G1_GEN = (bls.G1_GEN[0], bls.G1_GEN[1], 1)
BLS_X = 0xD201000000010000  # |x| of the BLS12-381 parameter
G1_COFACTOR = 0x396C8C005555E1568C00AAAB0000AAAB


# ---- off-subgroup G1 points ----------------------------------------------------------------------------------------


def curve_point(rng):
    """A uniformly random point of E(Fq): almost never in G1."""
    while True:
        x = rng.randrange(bls.P)
        y = bls.fq_sqrt(x**3 + 4)
        if y is not None:
            return (x, y, 1)


def in_g1(pt) -> bool:
    return bls.g1_mul_raw(pt, R) is None


@lru_cache(maxsize=None)
def torsion_point(order: int):
    """A point of E(Fq) of the given prime order dividing the cofactor (3, 11, 10177, ...)."""
    rest = G1_COFACTOR * R
    while rest % order == 0:
        rest //= order
    rng = random.Random(order)
    while True:
        t = bls.g1_mul_raw(curve_point(rng), rest)  # in the order-Sylow subgroup (Z_11 x Z_11 for 11, not cyclic)
        while t is not None and bls.g1_mul_raw(t, order) is not None:
            t = bls.g1_mul_raw(t, order)
        if t is not None:
            return bls.g1_to_affine(t) + (1,)


def scott_in_g1(pt) -> bool:
    """The device's membership test restated (Scott, ePrint 2021/1130): [x^2]P == (beta^2 X, -Y)."""
    a = bls.g1_to_affine(pt)
    if a is None:
        return True
    beta = next(b for b in (pow(c, (bls.P - 1) // 3, bls.P) for c in range(2, 10)) if b != 1)
    if not bls.g1_eq((beta * a[0] % bls.P, a[1], 1), bls.g1_mul_raw(pt, BLS_X * BLS_X - 1)):
        beta = beta * beta % bls.P  # the cube root whose eigenvalue on G1 is lambda = x^2 - 1 (msm.cuh glv_beta)
    return bls.g1_eq(bls.g1_mul_raw(pt, BLS_X * BLS_X), (beta * beta * a[0] % bls.P, (-a[1]) % bls.P, 1))


def membership_points(n_random: int = 12):
    """G1 points, every prime torsion order of the cofactor alone and shifted by G1 points, random curve points, cleared points."""
    rng = random.Random(3)
    pts = [G1_GEN, bls.g1_mul(G1_GEN, rng.randrange(R))]
    for order in (3, 11, 10177, 859267, 52437899):
        t = torsion_point(order)
        pts += [t, bls.g1_add(t, G1_GEN), bls.g1_add(t, bls.g1_mul(G1_GEN, rng.randrange(R)))]
    pts += [curve_point(rng) for _ in range(n_random)]
    pts += [bls.g1_mul_raw(curve_point(rng), G1_COFACTOR) for _ in range(3)]  # cleared: in G1
    return pts


def subgroup_test_matches_order(n_random: int = 12) -> None:
    """The membership test agrees with [r]P == O on G1 points, every small torsion order, shifted points and random points."""
    for pt in membership_points(n_random):
        assert scott_in_g1(pt) == in_g1(pt), bls.g1_to_affine(pt)
    rng = random.Random(4)
    # and the endomorphism split the device uses is wrong off G1: the reason the membership test exists
    p, k = curve_point(rng), rng.randrange(R)
    k2, k1 = divmod(k, BLS_X * BLS_X - 1)
    beta = next(b for b in (pow(c, (bls.P - 1) // 3, bls.P) for c in range(2, 10)) if b != 1)
    split = [bls.g1_add(bls.g1_mul_raw(p, k1), bls.g1_mul_raw((b * p[0] % bls.P, p[1], 1), k2)) for b in (beta, beta * beta % bls.P)]
    assert not any(bls.g1_eq(s, bls.g1_mul_raw(p, k)) for s in split)


def off_subgroup_mix(n: int, seed: int):
    """n affine points: SRS points, random curve points outside G1, SRS points shifted by 3- and 11-torsion, pure 3- and
    11-torsion points, infinity."""
    srs = rp.load_srs()
    rng = random.Random(seed)
    t3, t11 = torsion_point(3), torsion_point(11)
    out = []
    for i in range(n):
        base = (srs.g1[i % len(srs.g1)][0], srs.g1[i % len(srs.g1)][1], 1)
        kind = i % 5
        pt = base if kind == 0 else curve_point(rng) if kind == 1 else bls.g1_add(base, t3) if kind == 2 else bls.g1_add(base, t11) if kind == 3 else None
        if kind == 4 and i % 10 != 4:
            pt = curve_point(rng)
        if i % 7 == 6:  # pure small-order points: multiples of them reach infinity inside any window table
            pt = t3 if i % 14 == 6 else t11
        out.append(bls.g1_to_affine(pt) if pt is not None else None)
    return out


def enc96(a) -> bytes:
    return bls.g1_serialize(None if a is None else (a[0], a[1], 1))


def exact_msm(points, scalars):
    acc = None
    for a, k in zip(points, scalars):
        if a is not None:
            acc = bls.g1_add(acc, bls.g1_mul_raw((a[0], a[1], 1), k))
    return acc


def msm_off_subgroup(ctx, sizes, pool=None) -> None:
    """dr_g1_msm (and EnginePool.g1_msm) on points outside G1 against sum k_i * P_i, canonical scalars (< r)."""
    for n in sizes:
        pts = off_subgroup_mix(n, n)
        rng = random.Random(n + 1)
        ks = [rng.randrange(R) for _ in range(n)]
        if n > 2:
            ks[1], ks[2] = 1, R - 1
        want = bls.g1_serialize(exact_msm(pts, ks))
        # the C oracle MSM makes no subgroup assumption (integer windows, Jacobian): it agrees where it is defined
        if all(p is not None for p in pts):
            assert bls.g1_serialize(bls.g1_msm(pts, ks)) == want
        blob = b"".join(enc96(p) for p in pts)
        assert ctx.g1_msm(blob, ks) == want, n
        if pool is not None:
            assert pool.g1_msm(blob, ks, min_points_per_device=max(1, n // 3)) == want, n


def pairing_off_subgroup(ctx) -> None:
    """dr_pairing_check_batch with first arguments outside G1 against the oracle's Miller loop + final exponentiation."""
    rng = random.Random(9)
    srs = rp.load_srs()
    g2, g2tau = srs.g2
    tau_g = (srs.g1[1][0], srs.g1[1][1], 1)
    t3 = torsion_point(3)
    cases = [
        (bls.g1_add(G1_GEN, t3), g2, bls.g1_add(G1_GEN, t3), g2),
        (bls.g1_add(tau_g, t3), g2, G1_GEN, g2tau),
        (curve_point(rng), g2tau, G1_GEN, g2),
    ]
    expect = []
    for a1, b1, a2, b2 in cases:
        expect.append(bls.final_verify(bls.miller_loop(b1, bls.g1_to_affine(a1)), bls.miller_loop(b2, bls.g1_to_affine(a2))))
    got = ctx.pairing_check(
        b"".join(bls.g1_serialize(c[0]) for c in cases), b"".join(bls.g2_serialize(c[1]) for c in cases),
        b"".join(bls.g1_serialize(c[2]) for c in cases), b"".join(bls.g2_serialize(c[3]) for c in cases),
    )  # fmt: skip
    assert got == expect


# ---- oracle verdicts -------------------------------------------------------------------------------------------------


def pedersen_verdict(suite, proof: bytes, alpha: bytes, ad: bytes) -> int:
    try:
        p = ovrf.PedersenProof.decode(proof)
    except ValueError:
        return 2
    return int(ovrf.pedersen_verify(suite, p, alpha, ad))


def tiny_verdict(suite, pk: bytes, proof: bytes, alpha: bytes, ad: bytes) -> int:
    try:
        return int(ovrf.tiny_verify(suite, ovrf.TinyProof.decode(proof), pk, alpha, ad))
    except ValueError:
        return 2


def thin_verdict(suite, pk: bytes, proof: bytes, alpha: bytes, ad: bytes) -> int:
    try:
        return int(ovrf.thin_verify(suite, ovrf.ThinProof.decode(proof), pk, alpha, ad))
    except ValueError:
        return 2


class RingOracle:
    """Ring verdicts of the oracle for one ring, with explicit batching coefficients (the ones the device is given)."""

    def __init__(self, keys, params: rp.Params):
        self.params = params
        self.ring = rp.Ring(keys, params)
        self.root = rp.RingRoot.from_ring(self.ring, params)
        self.fixed = (self.root.px.commitment, self.root.py.commitment, self.root.s.commitment)
        self.prefix = self.root.transcript_prefix()
        self._parts = {}

    def parts(self, proof: bytes, alpha: bytes, ad: bytes):
        """(status, linear verifications): status 2 = decode raises, 0 = Pedersen part rejected, 1 = Pedersen part accepted."""
        key = (proof, alpha, ad)
        if key not in self._parts:
            try:
                p = ovrf.RingVrfProof.decode(proof)
            except ValueError:
                self._parts[key] = (2, None)
            else:
                ok = ovrf.pedersen_verify(self.params.suite, p.pedersen, alpha, ad)
                lin = rp.linear_verifications(self.params, self.fixed, self.prefix, p.pedersen.blinded_pk, p.ring)
                self._parts[key] = (int(ok), lin)
        return self._parts[key]

    def verdict(self, proof: bytes, alpha: bytes, ad: bytes, coeffs) -> int:
        st, lin = self.parts(proof, alpha, ad)
        if st != 1:
            return st
        return int(rp.batch_verify_linear(self.root.srs, lin, list(coeffs)))

    def aggregate(self, proofs, alphas, ads, coeffs):
        """(per-item decode / Pedersen status, all_ok) of the folded check, as dr_ring_verify_batch reports them."""
        parts = [self.parts(p, a, d) for p, a, d in zip(proofs, alphas, ads)]
        status = [st for st, _ in parts]
        if any(st != 1 for st in status):
            return status, False
        lin = [v for _, ls in parts for v in ls]
        return status, bool(rp.batch_verify_linear(self.root.srs, lin, list(coeffs)))


# ---- field mutations -------------------------------------------------------------------------------------------------


def _g1c(pt) -> bytes:
    return bls.g1_compress(pt)


@lru_cache(maxsize=1)
def _off_curve_x() -> bytes:
    x = 5
    while bls.fq_sqrt(x**3 + 4) is not None:
        x += 1
    out = bytearray(x.to_bytes(48, "big"))
    out[0] |= 0x80
    return bytes(out)


def g1_mutations(field: bytes, sibling: bytes):
    """(name, 48 bytes) replacements of a compressed G1 field."""
    pt = bls.g1_decompress(field)
    flip = bytearray(field)
    flip[47] ^= 1
    neg = bytearray(field)
    neg[0] ^= 0x20
    uncomp = bytearray(field)
    uncomp[0] &= 0x7F
    inf_flag = bytearray(_g1c(None))
    inf_flag[0] |= 0x20
    inf_tail = bytearray(_g1c(None))
    inf_tail[47] = 1
    x_ge_p = bytearray(bls.P.to_bytes(48, "big"))
    x_ge_p[0] |= 0x80
    return [
        ("bit_flip", bytes(flip)), ("generator", _g1c(G1_GEN)), ("negated", bytes(neg)), ("sibling", sibling),
        ("infinity", _g1c(None)), ("infinity_flag_bits", bytes(inf_flag)), ("infinity_tail_bits", bytes(inf_tail)),
        ("compression_bit_cleared", bytes(uncomp)), ("x_ge_p", bytes(x_ge_p)), ("x_off_curve", _off_curve_x()),
        ("outside_g1", _g1c(curve_point(random.Random(len(field) + field[5])))), ("plus_order3", _g1c(bls.g1_add(pt, torsion_point(3)))),
        ("order3", _g1c(torsion_point(3))), ("order11", _g1c(torsion_point(11))),
    ]  # fmt: skip


def fr_mutations(field: bytes, modulus: int):
    """(name, 32 bytes) replacements of a little-endian scalar field (BLS12-381 Fr or the Bandersnatch scalar field)."""
    v = int.from_bytes(field, "little")
    le = lambda x: x.to_bytes(32, "little")  # noqa: E731
    return [("plus_one", le((v + 1) % (1 << 256))), ("m_minus_v", le((modulus - v) % modulus)), ("zero", le(0)),
            ("modulus", le(modulus)), ("modulus_plus_one", le(modulus + 1)), ("all_ones", le((1 << 256) - 1))]  # fmt: skip


def fn_mutations(field: bytes):
    """Bandersnatch scalar field: +1, 0, n, n + 1, 2^256 - 1."""
    return [(m, x) for m, x in fr_mutations(field, bs.N) if m != "m_minus_v"]


@lru_cache(maxsize=1)
def _te_specials():
    enc = bs.point_to_string
    out = {"identity": enc(bs.IDENTITY), "zero_minus_one": enc((0, bs.P - 1)), "other_point": enc(bs.mul(bs.GENERATOR, 12345))}
    # No point of order 4 has an affine encoding: those are (+-1/sqrt(a), 0), and a = -5 is not a square, or lie at infinity.
    # The 2-torsion shift below is the only small-order component a 32-byte point can carry.
    assert bs.fr_sqrt(pow(bs.A, -1, bs.P)) is None
    y_ge_p = bytearray(bs.P.to_bytes(32, "little"))
    out["y_ge_p"] = bytes(y_ge_p)
    y = 2
    while True:
        rhs = (bs.A - bs.D * y * y) % bs.P
        if rhs and bs.fr_sqrt((1 - y * y) * pow(rhs, -1, bs.P) % bs.P) is None:
            break
        y += 1
    out["off_curve_y"] = y.to_bytes(32, "little")
    return out


def te_mutations(field: bytes):
    """(name, 32 bytes) replacements of a Bandersnatch point field or public key."""
    pt = bs.string_to_point(field)
    sign = bytearray(field)
    sign[31] ^= 0x80
    out = list(_te_specials().items())
    out.append(("plus_2torsion", bs.point_to_string(bs.add(pt, (0, bs.P - 1)))))
    out.append(("sign_flipped", bytes(sign)))
    return out


def mutate(proof: bytes, off: int, value: bytes) -> bytes:
    return proof[:off] + value + proof[off + len(value) :]


RING_G1 = {"c_b": 192, "c_accip": 240, "c_accx": 288, "c_accy": 336, "c_q": 608, "phi_zeta": 688, "phi_zeta_omega": 736}
RING_FR = {"px_zeta": 384, "py_zeta": 416, "s_zeta": 448, "b_zeta": 480, "accip_zeta": 512, "accx_zeta": 544, "accy_zeta": 576, "l_zeta_omega": 656}
PED_TE = {"output": 0, "blinded_pk": 32, "r": 64, "ok": 96}
PED_FN = {"s": 128, "sb": 160}


def pedersen_mutants(proof: bytes, te=PED_TE.items(), fn=PED_FN.items()):
    """(label, proof) for the four points and two scalars of a Pedersen proof (the first 192 bytes of a Ring VRF proof)."""
    out = []
    for name, off in te:
        out += [(f"{name}:{m}", mutate(proof, off, v)) for m, v in te_mutations(proof[off : off + 32])]
    for name, off in fn:
        out += [(f"{name}:{m}", mutate(proof, off, v)) for m, v in fn_mutations(proof[off : off + 32])]
    return out


def ring_mutants(proof: bytes, one_per_type: bool = False):
    """(label, proof) for every field of a 784-byte Ring VRF proof; one_per_type keeps one field of each kind."""
    g1 = list(RING_G1.items())[-1:] if one_per_type else RING_G1.items()
    frs = list(RING_FR.items())[-1:] if one_per_type else RING_FR.items()
    te = list(PED_TE.items())[1:2] if one_per_type else PED_TE.items()
    fn = list(PED_FN.items())[:1] if one_per_type else PED_FN.items()
    out = []
    for name, off in g1:
        sibling_off = RING_G1["c_b"] if off != RING_G1["c_b"] else RING_G1["c_q"]
        out += [(f"{name}:{m}", mutate(proof, off, v)) for m, v in g1_mutations(proof[off : off + 48], proof[sibling_off : sibling_off + 48])]
    for name, off in frs:
        out += [(f"{name}:{m}", mutate(proof, off, v)) for m, v in fr_mutations(proof[off : off + 32], R)]
    return out + pedersen_mutants(proof, te, fn)


def coeffs_random(n: int, seed: int) -> list[int]:
    rng = random.Random(seed)
    return [rng.randrange(1, R) for _ in range(2 * n)]


# ---- ring sweep ---------------------------------------------------------------------------------------------------------


def _ring_vector(prefix: str, index: int = 0):
    v = load(prefix + "_ring.json")[index]
    return v, split_keys(hx(v, "ring_pks")), hx(v, "alpha"), hx(v, "ad"), ring_proof_bytes(v)


def ring_tamper_sweep(srs, full_sha: bool = True, aggregate_sample: int | None = None) -> None:
    """Every field of the ring-8 reference proof (N = 512): SHA-512 in full, SHAKE128 one field per type."""
    for suite, prefix in SUITES:
        _, keys, alpha, ad, proof = _ring_vector(prefix)
        params = rp.Params(test_vectors=True, suite=suite)
        ring_sweep_one(srs, keys, params, alpha, ad, proof, one_per_type=(suite is not bs.SHA512) or not full_sha, aggregate_sample=aggregate_sample)


def ring1023_tamper_sweep(srs) -> None:
    """The same sweep on a proof produced by the unmodified reference at ring 1023 / N = 2048."""
    from tests.helpers import bench_ring_keys

    _, _, keys = bench_ring_keys(1023)
    e = load("ring1023_reference.json")["proofs_blinded"][0]
    ring_sweep_one(srs, keys, rp.Params.from_ring_size(1023), bytes.fromhex(e["alpha"]), bytes.fromhex(e["ad"]), bytes.fromhex(e["proof"]))


def ring_sweep_one(srs, keys, params, alpha: bytes, ad: bytes, proof: bytes, one_per_type: bool = False, aggregate_sample: int | None = None) -> None:
    """Per item (coefficients (1, random)), then every decodable mutant folded between two valid proofs through the
    13-multiplication route and the two-MSM route; aggregate_sample keeps that many of the opening / off-subgroup mutants."""
    oracle = RingOracle(keys, params)
    ring = native_ring(srs, keys, params)
    mutants = ring_mutants(proof, one_per_type=one_per_type)
    coeffs = []
    for i in range(len(mutants)):
        coeffs += [1, random.Random(i).randrange(1, R)]
    got, _ = ring.verify_batch([alpha] * len(mutants), [ad] * len(mutants), [m for _, m in mutants], coeffs)
    for i, (label, m) in enumerate(mutants):
        assert got[i] == oracle.verdict(m, alpha, ad, coeffs[2 * i : 2 * i + 2]), (label, got[i])
    interesting = [(label, m) for label, m in mutants if oracle.parts(m, alpha, ad)[0] != 2]
    if aggregate_sample is not None:
        interesting = [x for x in interesting if "phi" in x[0] or "outside" in x[0] or "order" in x[0]][:aggregate_sample]
    lib = ring.ctx.library.lib
    for i, (label, m) in enumerate(interesting):
        items = [proof, m, proof]
        co = coeffs_random(3, 100 + i)
        want = oracle.aggregate(items, [alpha] * 3, [ad] * 3, co)
        for threshold in (8192, 1):
            lib.dr_ring_verify_set_msm_threshold(threshold)
            try:
                got_v, got_ok = ring.verify_batch([alpha] * 3, [ad] * 3, items, co, aggregate=True)
            finally:
                lib.dr_ring_verify_set_msm_threshold(8192)
            assert (got_v, bool(got_ok)) == (want[0], want[1]), (label, threshold)
    ring.close()


# ---- VRF sweeps ---------------------------------------------------------------------------------------------------------


def vrf_tamper_sweep(ctx, suites=SUITES) -> None:
    """Tiny (O | c | s), Thin (O | R | s) and Pedersen proofs and the public keys, every field mutated, against the oracle."""
    for suite, prefix in suites:
        su = suite_struct(suite)
        v = load(prefix + "_pedersen.json")[0]
        alpha, ad = hx(v, "alpha"), hx(v, "ad")
        proof = hx(v, "gamma", "proof_pk_com", "proof_r", "proof_ok", "proof_s", "proof_sb")
        muts = [m for _, m in pedersen_mutants(proof)]
        got = ctx.pedersen_verify(su, [alpha] * len(muts), [ad] * len(muts), muts)
        assert got == [pedersen_verdict(suite, m, alpha, ad) for m in muts], prefix
        v = load(prefix + "_tiny.json")[0]
        alpha, ad, pk = hx(v, "alpha"), hx(v, "ad"), hx(v, "pk")
        proof = hx(v, "gamma", "proof_c", "proof_s")
        cases = [(pk, mutate(proof, 0, x)) for _, x in te_mutations(proof[:32])]
        c = int.from_bytes(proof[32:48], "little")
        cases += [(pk, mutate(proof, 32, x.to_bytes(16, "little"))) for x in ((c + 1) % (1 << 128), 0, (1 << 128) - 1)]
        cases += [(pk, mutate(proof, 48, x)) for _, x in fn_mutations(proof[48:])]
        cases += [(x, proof) for _, x in te_mutations(pk)]
        got = ctx.tiny_verify(su, [c[0] for c in cases], [alpha] * len(cases), [ad] * len(cases), [c[1] for c in cases])
        assert got == [tiny_verdict(suite, k, p, alpha, ad) for k, p in cases], prefix
        # Thin: SHA-512 vectors; the SHAKE128 proof comes from the oracle prover
        if suite is bs.SHA512:
            v = load(prefix + "_thin.json")[0]
            alpha, ad, pk = hx(v, "alpha"), hx(v, "ad"), hx(v, "pk")
            proof = hx(v, "gamma", "proof_r", "proof_s")
        else:
            proof = ovrf.thin_prove(suite, alpha, hx(v, "sk"), ad).encode()
        cases = [(pk, mutate(proof, off, x)) for off in (0, 32) for _, x in te_mutations(proof[off : off + 32])]
        cases += [(pk, mutate(proof, 64, x)) for _, x in fn_mutations(proof[64:])]
        cases += [(x, proof) for _, x in te_mutations(pk)]
        got = ctx.thin_verify(su, [c[0] for c in cases], [alpha] * len(cases), [ad] * len(cases), [c[1] for c in cases])
        assert got == [thin_verdict(suite, k, p, alpha, ad) for k, p in cases], prefix


def vrf_tamper_sweep_both_kernels(ctx, suites=SUITES) -> None:
    lib = ctx.library.lib
    vrf_tamper_sweep(ctx, suites)
    lib.dr_vrf_verify_set_coop_threshold(0)
    try:
        vrf_tamper_sweep(ctx, suites)
    finally:
        lib.dr_vrf_verify_set_coop_threshold(8192)


# ---- batch binding ------------------------------------------------------------------------------------------------------


@lru_cache(maxsize=1)
def _signers(count: int = 8):
    return [tr.secret_from_seed(bs.SHA512, seed("adversarial-signer", i)) for i in range(count)]


def distinct_proofs(srs, n: int = 5):
    """n valid ring proofs over one ring of 8, each by a different signer for a different input / ad."""
    params = rp.Params()
    signers = _signers()
    keys = [pk for pk, _ in signers]
    ring = native_ring(srs, keys, params)
    alphas = [b"adversarial-input-%d" % i for i in range(n)]
    ads = [b"ad-%d" % (i * 7) for i in range(n)]
    proofs = []
    for i in range(n):
        got, st = ring.prove_batch([alphas[i]], [ads[i]], [signers[i][1]], [i])
        assert st == [0]
        proofs.append(got[0])
    return ring, keys, params, alphas, ads, proofs


def batch_binding(srs, n: int = 5, pool_ring=None) -> None:
    """Recombined batches: inputs / ads rotated by one, ring halves and Pedersen halves rotated between proofs.  Each item's
    verdict is the oracle's at its own index; a tampered item inside a folded batch makes it fail."""
    ring, keys, params, alphas, ads, proofs = distinct_proofs(srs, n)
    oracle = RingOracle(keys, params)
    co = coeffs_random(n, 11)
    rot = lambda xs: xs[1:] + xs[:1]  # noqa: E731
    batches = {
        "honest": (alphas, ads, proofs),
        "inputs_rotated": (rot(alphas), ads, proofs),
        "ads_rotated": (alphas, rot(ads), proofs),
        "ring_halves_rotated": (alphas, ads, [p[:192] + q[192:] for p, q in zip(proofs, rot(proofs))]),
        "pedersen_halves_rotated": (alphas, ads, [q[:192] + p[192:] for p, q in zip(proofs, rot(proofs))]),
    }
    for name, (a, d, p) in batches.items():
        want = [oracle.verdict(p[i], a[i], d[i], co[2 * i : 2 * i + 2]) for i in range(n)]
        assert want == ([1] * n if name == "honest" else [0] * n), name
        assert ring.verify_batch(a, d, p, co)[0] == want, name
        # one recombined item among honest ones, at every index, folded
        for i in (0, n // 2, n - 1):
            a2, d2, p2 = list(alphas), list(ads), list(proofs)
            a2[i], d2[i], p2[i] = a[i], d[i], p[i]
            agg = oracle.aggregate(p2, a2, d2, co)
            assert ring.verify_batch(a2, d2, p2, co, aggregate=True) == (agg[0], agg[1]) and agg[1] == (name == "honest"), (name, i)
            if pool_ring is not None:
                assert pool_ring(a2, d2, p2, co) == [oracle.verdict(p2[j], a2[j], d2[j], co[2 * j : 2 * j + 2]) for j in range(n)], (name, i)
    ring.close()
    return keys, alphas, ads, proofs


def wrong_ring_through_api(api, keys, alphas, ads, proofs) -> None:
    """A valid proof does not verify against a ring that differs in one key (the Python API compares ring roots)."""
    params = api.RingProofParams()
    cls = api.RingVRF[api.Bandersnatch]
    good = api.Ring(keys, params)
    other_keys = list(keys)
    other_keys[-1] = tr.secret_from_seed(bs.SHA512, seed("not-a-member"))[0]
    other = api.Ring(other_keys, params)
    assert cls.verify_batch(proofs, alphas, ads, good, api.RingRoot.from_ring(good, params)) == [1] * len(proofs)
    assert cls.verify_batch(proofs, alphas, ads, other, api.RingRoot.from_ring(other, params)) == [0] * len(proofs)


# ---- coefficient-exact openings -----------------------------------------------------------------------------------------


def _zeta(oracle: RingOracle, proof: bytes) -> int:
    rv = ovrf.RingVrfProof.decode(proof)
    return rp.verifier_challenges(oracle.prefix, rv.pedersen.blinded_pk, rv.ring)[1]


def _opening_shift(oracle: RingOracle, point: int, c: int):
    """c * (point * G - [tau]_1)"""
    tau_g = (oracle.root.srs.g1[1][0], oracle.root.srs.g1[1][1], 1)
    return bls.g1_mul(bls.g1_add(bls.g1_mul(G1_GEN, point), bls.g1_neg(tau_g)), c)


def _add_at(proof: bytes, off: int, pt) -> bytes:
    return proof[:off] + bls.g1_compress(bls.g1_add(bls.g1_decompress(proof[off : off + 48]), pt)) + proof[off + 48 :]


def forge_openings(oracle: RingOracle, proof: bytes, c1: int, c2: int) -> bytes:
    """phi_zeta + c2 (zeta w G - [tau]_1), phi_zeta_omega - c1 (zeta G - [tau]_1): e(lhs, [1]_2) == e(rhs, [tau]_2) still holds
    with exactly the coefficients (c1, c2), and the challenges do not move (the openings are not absorbed)."""
    z = _zeta(oracle, proof)
    out = _add_at(proof, 688, _opening_shift(oracle, z * oracle.params.omega % R, c2))
    return _add_at(out, 736, bls.g1_neg(_opening_shift(oracle, z, c1)))


def coefficient_exact_openings(srs) -> None:
    """A forgery built for one pair of coefficients: the device must accept exactly where the oracle does."""
    v, keys, alpha, ad, proof = _ring_vector("bandersnatch_sha-512_ell2")
    params = rp.Params(test_vectors=True)
    oracle = RingOracle(keys, params)
    ring = native_ring(srs, keys, params)
    rr = random.Random(21).randrange(2, R - 1)
    forged = forge_openings(oracle, proof, 1, rr)
    for co in ((1, rr), (1, rr + 1), (rr, 1)):
        want = oracle.verdict(forged, alpha, ad, co)
        assert want == (co == (1, rr))
        assert ring.verify_batch([alpha], [ad], [forged], list(co))[0] == [want], co
    forged11 = forge_openings(oracle, proof, 1, 1)  # caught only by a kernel that applies the caller's coefficients
    assert oracle.verdict(forged11, alpha, ad, (1, rr)) == 0
    assert ring.verify_batch([alpha], [ad], [forged11], [1, rr])[0] == [0]
    # across two proofs of one folded batch with coefficients (a0, b0, a1, b1): phi_zeta of proof 0 gets X1, phi_zeta_omega of
    # proof 1 gets X2; the folded check moves by a0 (zeta0 - tau) X1 + b1 (zeta1 w - tau) X2, which
    # X1 = b1 (zeta1 w G - [tau]_1), X2 = -a0 (zeta0 G - [tau]_1) cancel.  Each proof alone fails.
    co = [3, 5, 7, 11]
    a2, d2 = b"second", b"proof"
    p2, st = ring.prove_batch([a2], [d2], [hx(v, "sk")], [oracle.ring.index_of(hx(v, "pk"))])
    assert st == [0]
    p2 = p2[0]
    f1 = _add_at(proof, 688, _opening_shift(oracle, _zeta(oracle, p2) * params.omega % R, co[3]))
    f2 = _add_at(p2, 736, bls.g1_neg(_opening_shift(oracle, _zeta(oracle, proof), co[0])))
    want = oracle.aggregate([f1, f2], [alpha, a2], [ad, d2], co)
    assert want == ([1, 1], True)
    lib = ring.ctx.library.lib
    for threshold in (8192, 1):
        lib.dr_ring_verify_set_msm_threshold(threshold)
        try:
            assert ring.verify_batch([alpha, a2], [ad, d2], [f1, f2], co, aggregate=True) == ([1, 1], True), threshold
        finally:
            lib.dr_ring_verify_set_msm_threshold(8192)
    per_item = [oracle.verdict(f1, alpha, ad, co[:2]), oracle.verdict(f2, a2, d2, co[2:])]
    assert per_item == [0, 0] and ring.verify_batch([alpha, a2], [ad, d2], [f1, f2], co)[0] == per_item
    ring.close()
