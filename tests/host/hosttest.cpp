// Host-compiled copy of the product's __host__ __device__ math headers, exported as a small C
// library for CPU unit tests (tests/test_host_math.py compares it with the oracle).  Test
// infrastructure only: nothing in dot_ring_b200 loads this library.
#include <cstdint>
#include <cstring>

#include "../../dot_ring_b200/csrc/fp.cuh"
#include "../../dot_ring_b200/csrc/g1.cuh"
#include "../../dot_ring_b200/csrc/hash.cuh"
#include "../../dot_ring_b200/csrc/msm.cuh"
#include "../../dot_ring_b200/csrc/te.cuh"

using namespace dr;

static Fq fq_in(const uint8_t* b) {
    Fq r;
    fq_from_be_bytes_raw(r, b);
    return r.to_mont();
}
static void fq_out(uint8_t* b, const Fq& x) { fq_to_be_bytes_raw(b, x.from_mont()); }
static Fr fr_in(const uint8_t* b) {
    Fr r;
    fr_from_le_bytes_raw(r, b);
    return r.to_mont();
}
static void fr_out(uint8_t* b, const Fr& x) { fr_to_le_bytes_raw(b, x.from_mont()); }

extern "C" {
// op: 0 mul, 1 add, 2 sub, 3 inv(a), 4 sqrt(a) (returns 0 if none), 5 sqr
int ht_fq_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out) {
    Fq x = fq_in(a), y = fq_in(b), r = Fq::zero();
    int ok = 1;
    switch (op) {
        case 0: r = x * y; break;
        case 1: r = x + y; break;
        case 2: r = x - y; break;
        case 3: r = x.inv(); break;
        case 4: ok = fq_sqrt(r, x); break;
        case 5: r = x.sqr(); break;
    }
    fq_out(out, r);
    return ok;
}
int ht_fr_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out) {
    Fr x = fr_in(a), y = fr_in(b), r = Fr::zero();
    int ok = 1;
    switch (op) {
        case 0: r = x * y; break;
        case 1: r = x + y; break;
        case 2: r = x - y; break;
        case 3: r = x.inv(); break;
        case 4: ok = fr_sqrt(r, x); break;
        case 5: r = x.sqr(); break;
        case 6: ok = fr_is_square(x); break;
    }
    fr_out(out, r);
    return ok;
}
// field: 0 Fq (48-byte big-endian), 1 Fr (32-byte little-endian).  out = inv() (division steps), out2 = Fermat inverse, out3 = Kaliski's
// binary inverse; returns the Legendre symbol
int ht_inv_and_legendre(int field, const uint8_t* a, uint8_t* out, uint8_t* out2, uint8_t* out3) {
    if (field == 0) {
        Fq x = fq_in(a);
        fq_out(out, x.inv());
        fq_out(out2, x.inv_fermat());
        fq_out(out3, x.inv_kaliski());
        return x.legendre();
    }
    Fr x = fr_in(a);
    fr_out(out, x.inv());
    fr_out(out2, x.inv_fermat());
    fr_out(out3, x.inv_kaliski());
    return x.legendre();
}
// prime-subgroup membership of an on-curve point, both ways: bit 0 = 2-descent (two Legendre symbols), bit 1 = multiplication by the order
int ht_te_subgroup(const uint8_t* xy64) {
    TEAffine p{fr_in(xy64), fr_in(xy64 + 32)};
    return (te_in_prime_subgroup(p) ? 1 : 0) | (te_in_prime_subgroup_by_order(p) ? 2 : 0);
}
// GLV: out32 = encode(k * P) through te_mul_glv; split16x2 = |k1| (16 bytes LE) | |k2| (16 bytes LE); returns sign bits (1: k1 < 0, 2: k2 < 0)
int ht_te_mul_glv(const uint8_t* point32, const uint8_t* k32, uint8_t* out32, uint8_t* split32) {
    TEAffine p;
    if (!te_decode(p, point32)) return -1;
    uint32_t k[8], k1[8], k2[8];
    for (int i = 0; i < 8; i++) k[i] = (uint32_t)k32[4 * i] | ((uint32_t)k32[4 * i + 1] << 8) | ((uint32_t)k32[4 * i + 2] << 16) | ((uint32_t)k32[4 * i + 3] << 24);
    bool n1, n2;
    te_glv_split(k, k1, n1, k2, n2);
    for (int i = 4; i < 8; i++)
        if (k1[i] | k2[i]) return -2;  // halves must fit 128 bits
    for (int i = 0; i < 4; i++)
        for (int b = 0; b < 4; b++) {
            split32[4 * i + b] = (uint8_t)(k1[i] >> (8 * b));
            split32[16 + 4 * i + b] = (uint8_t)(k2[i] >> (8 * b));
        }
    te_encode(out32, te_to_affine(te_mul_glv(p, k)));
    return (n1 ? 1 : 0) | (n2 ? 2 : 0);
}
// reduce len bytes (little-endian) mod the Bandersnatch group order; out 32 LE
void ht_fn_from_bytes_mod(const uint8_t* in, int len, uint8_t* out) {
    Fn x = fp_from_le_bytes_mod<Fn>(in, len).from_mont();
    for (int i = 0; i < 8; i++)
        for (int b = 0; b < 4; b++) out[4 * i + b] = (uint8_t)(x.v[i] >> (8 * b));
}
// s = k + c*x mod n (all 32-byte LE canonical)
void ht_fn_muladd(const uint8_t* k, const uint8_t* c, const uint8_t* x, uint8_t* out) {
    Fn r = fp_from_le_bytes_mod<Fn>(k, 32) + fp_from_le_bytes_mod<Fn>(c, 32) * fp_from_le_bytes_mod<Fn>(x, 32);
    r = r.from_mont();
    for (int i = 0; i < 8; i++)
        for (int b = 0; b < 4; b++) out[4 * i + b] = (uint8_t)(r.v[i] >> (8 * b));
}

int ht_g1_decode(const uint8_t* in, int len, uint8_t* out96) {
    G1Affine a;
    if (!g1_decode(a, in, len)) return 0;
    g1_serialize(out96, a);
    return 1;
}
int ht_g1_in_subgroup(const uint8_t* in96) {
    G1Affine a;
    if (!g1_decode(a, in96, 96)) return -1;
    return g1_in_subgroup(a) ? 1 : 0;
}

void ht_g1_compress(const uint8_t* in96, uint8_t* out48) {
    G1Affine a;
    g1_decode(a, in96, 96);
    g1_compress(out48, a);
}
// out = a + b, inputs/outputs 96-byte uncompressed; mode 0: XYZZ+XYZZ, 1: mixed
void ht_g1_add(const uint8_t* a96, const uint8_t* b96, int mode, uint8_t* out96) {
    G1Affine a, b;
    g1_decode(a, a96, 96);
    g1_decode(b, b96, 96);
    G1 acc = G1::from_affine(a);
    if (mode == 1) {
        g1_madd(acc, b);
    } else {
        // make b projective with a non-trivial ZZ by doubling and adding back -b ... keep simple: b as-is
        G1 pb = G1::from_affine(b);
        g1_add(acc, pb);
    }
    g1_serialize(out96, g1_to_affine(acc));
}
// out = k * a via double-and-add on XYZZ (exercises dbl/add with general Z)
void ht_g1_mul(const uint8_t* a96, const uint8_t* k32le, uint8_t* out96) {
    G1Affine a;
    g1_decode(a, a96, 96);
    G1 acc = G1::inf();
    G1 base = G1::from_affine(a);
    for (int i = 0; i < 256; i++) {
        if ((k32le[i >> 3] >> (i & 7)) & 1) g1_add(acc, base);
        base = g1_dbl(base);
    }
    g1_serialize(out96, g1_to_affine(acc));
}
// out = k * a by g1_mul_limbs (4-bit windows over an XYZZ table: the verifier's multiplication for points outside G1)
void ht_g1_mul_limbs(const uint8_t* a96, const uint8_t* k32le, uint8_t* out96) {
    G1Affine a;
    g1_decode(a, a96, 96);
    uint32_t k[8];
    memcpy(k, k32le, 32);
    g1_serialize(out96, g1_to_affine(g1_mul_limbs(G1::from_affine(a), k)));
}
// out = k * a using mixed additions only (left-to-right)
void ht_g1_mul_mixed(const uint8_t* a96, const uint8_t* k32le, uint8_t* out96) {
    G1Affine a;
    g1_decode(a, a96, 96);
    G1 acc = G1::inf();
    for (int i = 255; i >= 0; i--) {
        acc = g1_dbl(acc);
        if ((k32le[i >> 3] >> (i & 7)) & 1) g1_madd(acc, a);
    }
    g1_serialize(out96, g1_to_affine(acc));
}

int ht_te_decode(const uint8_t* in32, int checked, uint8_t* xy64) {
    TEAffine p;
    bool ok = checked ? te_decode_checked(p, in32) : te_decode(p, in32);
    if (!ok) return 0;
    fr_out(xy64, p.x);
    fr_out(xy64 + 32, p.y);
    return 1;
}
void ht_te_mul(const uint8_t* in32, const uint8_t* k32le, uint8_t* out32) {
    TEAffine p;
    te_decode(p, in32);
    uint32_t k[8];
    for (int i = 0; i < 8; i++) k[i] = (uint32_t)k32le[4 * i] | ((uint32_t)k32le[4 * i + 1] << 8) | ((uint32_t)k32le[4 * i + 2] << 16) | ((uint32_t)k32le[4 * i + 3] << 24);
    te_encode(out32, te_to_affine(te_mul_raw(p, k, 8)));
}
void ht_te_msm(const uint8_t* pts32, const uint8_t* ks32, int n, uint8_t* out32) {
    TEAffine p[3];
    uint32_t k[3][8];
    for (int j = 0; j < n; j++) {
        te_decode(p[j], pts32 + 32 * j);
        for (int i = 0; i < 8; i++) {
            const uint8_t* s = ks32 + 32 * j + 4 * i;
            k[j][i] = (uint32_t)s[0] | ((uint32_t)s[1] << 8) | ((uint32_t)s[2] << 16) | ((uint32_t)s[3] << 24);
        }
    }
    te_encode(out32, te_to_affine(te_msm_small(p, k, n)));
}
// u0, u1: 48-byte big-endian hash_to_field outputs
void ht_te_ell2(const uint8_t* u0_be48, const uint8_t* u1_be48, uint8_t* out32) {
    te_encode(out32, te_encode_to_curve_from_u(fr_from_be48_mod(u0_be48), fr_from_be48_mod(u1_be48)));
}
// One batched-affine round (msm.cuh: affine_round) over `n` points given as 96-byte encodings (pairs (0,1), (2,3), ...):
// out = n/2 sums.  Exercises the exceptional cases of the affine law that real SRS data never produces.
void ht_affine_round(const uint8_t* in96, int n, uint8_t* out96) {
    std::vector<G1Affine> pts(n);
    for (int i = 0; i < n; i++) g1_decode(pts[i], in96 + 96 * i, 96);
    const uint32_t pairs = n / 2;
    std::vector<Fq> prefix((size_t)pairs * 32);
    std::vector<G1Affine> out((size_t)pairs * 32);
    affine_round(pairs, 0, [&](uint32_t j) { return pts[j]; }, [&](uint32_t j) { return pts[j].x; }, prefix.data(), out.data());
    for (uint32_t i = 0; i < pairs; i++) g1_serialize(out96 + 96 * i, out[(size_t)i * 32]);
}
void ht_sha512(const uint8_t* msg, uint32_t len, uint8_t* out64) {
    Sha512 s;
    s.init();
    s.update(msg, len);
    s.final(out64);
}
void ht_shake128(const uint8_t* msg, uint32_t len, uint8_t* out, uint32_t outlen) {
    Shake128 s;
    s.init();
    s.absorb(msg, len);
    s.squeeze_snapshot(out, outlen);
}
}
