// Ring-proof prover kernels (batched over proofs).
//
// Device restatement of the reference prover pipeline:
//   dot_ring/ring_proof/columns/columns.py:111-167       witness columns b / acc_x / acc_y / acc_ip
//   dot_ring/ring_proof/constraints/constraints.py:43-151 4x LDE + constraints c1..c7
//   dot_ring/ring_proof/proof_builder.py:38-315           aggregation, quotient, linearisation, openings
//   dot_ring/ring_proof/polynomial/ops.py:170-224         Horner, divide by X^N - 1
//   dot_ring/ring_proof/pcs/utils.py:27-35                synthetic division
//   dot_ring/ring_proof/transcript/{transcript,phases}.py Fiat-Shamir (SHAKE128)
//   dot_ring/vrf/pedersen/vrf.py:86-126                   Pedersen VRF prove (SHA-512 transcripts)
// One proof is one row of every buffer; the 4N ("radix") domain is handled as four cosets of the
// N-domain (point 4i+j = w4^j * w^i is stored at [j*N + i]) so every transform is an N-point NTT
// that fits one CTA's shared memory, and the shifted row access i+4 (mod 4N) of the constraints
// becomes i+1 (mod N) inside a coset.
#pragma once
#include "g1.cuh"
#include "hash.cuh"
#include "msm.cuh"
#include "ntt.cuh"
#include "rt.cuh"
#include "te.cuh"
#include "te_coop.cuh"

namespace dr {

constexpr uint32_t SCALAR_BITS = 253;

// What a pass reads that depends only on the domain size N or on the suite, passed to kernels by value.  The ring's own data
// (keys, fixed columns, transcript prefix) is in RingTab, so that one pass can prove items of several rings.
struct RingDev {
    uint32_t N, logN, last;            // last = N - 4 (last accumulator row)
    const Fr* tw_fwd;                  // [N/2] w^k
    const Fr* tw_inv;                  // [N/2] w^-k
    const Fr* w4;                      // [4N]  w4^k
    const Fr* w4inv;                   // [4N]  w4^-k
    Fr n_inv;                          // 1/N
    Fr quarter;                        // 1/4
    Fr omega;                          // w
    Fr w_last;                         // w^(N-4)
    Fr tail[4];                        // coefficients of (X - w^(N-1))(X - w^(N-2))(X - w^(N-3))
    TEAffine seed, blinding_base, generator;
    const TEPre* g_tab;  // window tables of generator / blinding_base for te_mul_fixed (TeFixedTableBody)
    const TEPre* b_tab;
    uint32_t suite_id_len;
    uint8_t suite_id[32];
    uint32_t dst_len;
    uint8_t dst[64];  // hash-to-curve DST (without the trailing length byte)
    uint32_t hash_kind;  // 0: SHA-512 suite (XMD h2c, counter-mode squeeze), 1: SHAKE128 suite (XOF h2c, direct squeeze)
};

// One ring's device tables: an array of these is indexed by ProofState::ring.  The kernels that read them run one proof per
// block or per warp and resolve the entry there, before any branch on per-thread data.
struct RingTab {
    const TEAffine* nm;      // [N]   PK || padding || 2^i B || 4 x (0,0)
    const Fr* fixed_coef;    // [3][N]   px, py, s  coefficients
    const Fr* fixed_lde;     // [6][4N]  px, py, s, L_0, L_last, (x - w^last): coset layout
    const Shake128* prefix;  // ring transcript after the verifier key (root.py:54-71)
    uint32_t max_ring;
};

// The suite's transcript hash (primitives.py:26-55).  Absorb-only until squeezed; squeezing never disturbs the state, so a
// copy can keep absorbing.  SHA-512 suites squeeze in counter mode (primitives.py:165-174: seed = H(absorbed),
// block c = H(seed | le64(c))); the SHAKE128 suite squeezes the XOF directly.
struct VrfHash {
    uint32_t kind;
    union {
        Sha512 sha;
        Shake128 shake;
    };
    DR_HD void init(uint32_t k) {
        kind = k;
        if (kind == 0) sha.init();
        else shake.init();
    }
    DR_HD void update(const uint8_t* data, uint32_t len) {
        if (kind == 0) sha.update(data, len);
        else shake.absorb(data, len);
    }
    DR_HD void update_byte(uint8_t b) { update(&b, 1); }
    DR_HD_COLD void squeeze(uint8_t* out, uint32_t size) const {
        if (kind != 0) {
            shake.squeeze_snapshot(out, size);
            return;
        }
        Sha512 h = sha;
        uint8_t seed[64];
        h.final(seed);
        uint32_t done = 0;
        for (uint64_t c = 0; done < size; c++) {
            Sha512 b;
            b.init();
            b.update(seed, 64);
            uint8_t ctr[8];
            for (int i = 0; i < 8; i++) ctr[i] = (uint8_t)(c >> (8 * i));
            b.update(ctr, 8);
            uint8_t blk[64];
            b.final(blk);
            for (uint32_t i = 0; i < 64 && done < size; i++) out[done++] = blk[i];
        }
    }
};
// Per-proof state (one element of an array in HBM).
struct ProofState {
    uint32_t k;         // producer index
    uint32_t status;    // 0 ok; 1 = producer key does not match secret key / ring row
    uint32_t ring;      // entry of the call's RingTab array
    uint32_t t[8];      // Pedersen blinding factor, raw limbs
    Fr zk[12];          // blinding rows: b, accx, accy, accip (3 each), Montgomery
    TEAffine a0;        // seed + PK_k
    TEAffine s[SCALAR_BITS];  // accumulator after bit row j
    TEAffine relation;  // PK_k + t*B  (== Pedersen blinded key)
    Shake128 tr;        // ring transcript
    Fr alpha[7], zeta, nu[8];
    Fr evals[7];        // px, py, s, b, accip, accx, accy at zeta
    Fr lzw;             // L(zeta * w)
    G1Affine commits[7];  // C_b, C_accip, C_accx, C_accy, C_q, Phi_zeta, Phi_zeta_w
    uint8_t pedersen[192];
    // hand-over from the first half of the Pedersen prover (everything the ring proof needs) to the second half, which runs on a
    // side stream next to the ring-proof pipeline
    TEAffine vrf_input;  // hash-to-curve point
    VrfHash vrf_tr;      // VRF transcript after the blinded key
};

struct ProveInput {  // host-packed per proof
    uint32_t alpha_off, alpha_len, ad_off, ad_len;
    uint32_t k;
    uint32_t ring;  // entry of the call's RingTab array
    uint8_t sk[32];  // Ring VRF: the secret key; bare ring proof: the blinding factor t (both little-endian, below the group order)
};

// column index convention inside the prover buffers
enum { COL_B = 0, COL_ACCX = 1, COL_ACCY = 2, COL_ACCIP = 3 };

// ---- small helpers ---------------------------------------------------------------------------------
DR_HD void shake_absorb_label(Shake128& s, const char* label, uint32_t len) {
    s.absorb((const uint8_t*)label, len);
    s.absorb_be32(len);
}
DR_HD void shake_absorb_labeled_begin(Shake128& s, const char* label, uint32_t len) { shake_absorb_label(s, label, len); }
// challenge squeeze: 48 bytes big-endian mod r -> Montgomery Fr
DR_HD Fr shake_challenge_value(const Shake128& s) {
    uint8_t out[48];
    s.squeeze_snapshot(out, 48);
    return fr_from_be48_mod(out);
}
// transcript.py:109-136: prefix = label | be32(len) | "challenge"; after each squeeze absorb footer 00 00 00 09
DR_HD_COLD void shake_challenges(Shake128& s, const char* label, uint32_t len, Fr* out, int n) {
    for (int i = 0; i < n; i++) {
        shake_absorb_label(s, label, len);
        s.absorb((const uint8_t*)"challenge", 9);
        out[i] = shake_challenge_value(s);
        s.absorb_be32(9);
    }
}
DR_HD void shake_absorb_fr(Shake128& s, const Fr& x_mont) {
    uint8_t b[32];
    fr_to_le_bytes_raw(b, x_mont.from_mont());
    s.absorb(b, 32);
}
DR_HD void shake_absorb_g1(Shake128& s, const G1Affine& p) {
    uint8_t b[96];
    g1_serialize(b, p);
    s.absorb(b, 96);
}

DR_HD void vrf_squeeze(const VrfHash& st, uint8_t* out, uint32_t size) { st.squeeze(out, size); }
DR_HD void fn_to_le_bytes(uint8_t* out, const Fn& x_mont) {
    Fn x = x_mont.from_mont();
    for (int i = 0; i < 8; i++)
        for (int b = 0; b < 4; b++) out[4 * i + b] = (uint8_t)(x.v[i] >> (8 * b));
}
// primitives.py:66-82 `nonce`
DR_HD_COLD Fn vrf_nonce(const VrfHash& t, const Fn& secret) {
    VrfHash te = t;
    te.update_byte(0x10);
    uint8_t sb[32];
    fn_to_le_bytes(sb, secret);
    te.update(sb, 32);
    uint8_t secret_hash[64];
    vrf_squeeze(te, secret_hash, 64);
    VrfHash tn = t;
    tn.update_byte(0x11);
    tn.update(secret_hash, 64);
    uint8_t wide[48];
    vrf_squeeze(tn, wide, 48);
    return fp_from_le_bytes_mod<Fn>(wide, 48);
}
DR_HD void fn_raw_limbs(uint32_t* out, const Fn& x_mont) {
    Fn x = x_mont.from_mont();
    for (int i = 0; i < 8; i++) out[i] = x.v[i];
}
DR_HD_COLD TEAffine te_mul_fn(const TEAffine& p, const Fn& k) {  // p in the prime subgroup
    uint32_t kr[8];
    fn_raw_limbs(kr, k);
    return te_to_affine(te_mul_glv(p, kr));
}
DR_HD void sha_absorb_point(VrfHash& s, const TEAffine& p) {
    uint8_t b[32];
    te_encode(b, p);
    s.update(b, 32);
}

// expand_message_xmd(SHA-512) for 96 output bytes (curve.py:145-185; Z_pad = 48 bytes for this suite)
template <class S>
DR_HD_COLD void h2c_uniform_bytes(const S& rg, const uint8_t* msg, uint32_t msg_len, uint8_t* out96) {
    uint8_t dst_prime_len = (uint8_t)rg.dst_len;
    if (rg.hash_kind != 0) {  // expand_message_xof: SHAKE128(msg | I2OSP(96, 2) | DST | I2OSP(len(DST), 1))
        Shake128 x;
        x.init();
        x.absorb(msg, msg_len);
        uint8_t lib2[2] = {0, 96};
        x.absorb(lib2, 2);
        x.absorb(rg.dst, rg.dst_len);
        x.absorb_byte(dst_prime_len);
        x.squeeze_snapshot(out96, 96);
        return;
    }
    Sha512 h;
    h.init();
    uint8_t zero[48];
    for (int i = 0; i < 48; i++) zero[i] = 0;
    h.update(zero, 48);
    h.update(msg, msg_len);
    uint8_t lib[3] = {0, 96, 0};
    h.update(lib, 3);
    h.update(rg.dst, rg.dst_len);
    h.update_byte(dst_prime_len);
    uint8_t b0[64];
    h.final(b0);
    uint8_t prev[64];
    for (int blk = 1; blk <= 2; blk++) {
        Sha512 g;
        g.init();
        uint8_t x[64];
        for (int i = 0; i < 64; i++) x[i] = blk == 1 ? b0[i] : (uint8_t)(b0[i] ^ prev[i]);
        g.update(x, 64);
        g.update_byte((uint8_t)blk);
        g.update(rg.dst, rg.dst_len);
        g.update_byte(dst_prime_len);
        g.final(prev);
        for (int i = 0; i < 64 && 64 * (blk - 1) + i < 96; i++) out96[64 * (blk - 1) + i] = prev[i];
    }
}
template <class S>
DR_HD TEAffine vrf_encode_to_curve(const S& rg, const uint8_t* msg, uint32_t msg_len) {
    uint8_t u[96];
    h2c_uniform_bytes(rg, msg, msg_len, u);
    return te_encode_to_curve_from_u(fr_from_be48_mod(u), fr_from_be48_mod(u + 48));
}

// ---- A. Pedersen VRF prove (pedersen/vrf.py:86-126) -------------------------------------------------------
// First half: everything up to the blinded key, in two steps around the blinding-base multiplication so that the cooperative
// prover can run the multiplications on several lanes.
// Step 1: public key and output point (given in extended coordinates), VRF transcript, blinding factor.  Writes O into out192.
template <class S>
DR_HD_COLD void pedersen_begin_transcript(const S& rg, const Fn& x, const TEAffine& input, const TEExt& pk_ext, const TEExt& output_ext, const uint8_t* ad,
                                          uint32_t ad_len, uint8_t* out192, TEAffine& pk, uint32_t* blinding_raw, VrfHash& tr) {
    TEAffine output;
    te_to_affine2(pk_ext, output_ext, pk, output);
    // vrf_transcript (primitives.py:102-144) with one I/O pair
    tr.init(rg.hash_kind);
    tr.update(rg.suite_id, rg.suite_id_len);
    tr.update_byte(0x02);
    uint8_t le[8] = {1, 0, 0, 0, 0, 0, 0, 0};
    tr.update(le, 8);
    sha_absorb_point(tr, input);
    sha_absorb_point(tr, output);
    for (int i = 0; i < 8; i++) le[i] = i < 4 ? (uint8_t)(ad_len >> (8 * i)) : 0;
    tr.update(le, 8);
    tr.update(ad, ad_len);
    // blinding factor
    VrfHash tb = tr;
    tb.update_byte(0x12);
    Fn b = vrf_nonce(tb, x);
    fn_raw_limbs(blinding_raw, b);
    te_encode(out192, output);
}
// Step 2: blinded key Ybar = pk + b * B (b * B given), absorbed into the transcript.  Writes Ybar into out192 + 32.
DR_HD_COLD void pedersen_begin_blind(const TEAffine& pk, const TEExt& bB_ext, uint8_t* out192, TEAffine& blinded, VrfHash& tr) {
    blinded = te_to_affine(te_add(bB_ext, TEExt::from_affine(pk)));
    sha_absorb_point(tr, blinded);
    te_encode(out192 + 32, blinded);
}
// Writes O | Ybar into out192; returns the public key, the blinded key, the blinding factor and the transcript state the second
// half continues from.  `input` is the hash-to-curve point.
template <class S>
DR_HD_COLD void pedersen_prove_begin(const S& rg, const uint8_t* sk32, const TEAffine& input, const uint8_t* ad, uint32_t ad_len, uint8_t* out192, TEAffine& pk,
                                     TEAffine& blinded, uint32_t* blinding_raw, VrfHash& tr) {
    Fn x = fp_from_le_bytes_mod<Fn>(sk32, 32);
    uint32_t xr[8];
    fn_raw_limbs(xr, x);
    pedersen_begin_transcript(rg, x, input, te_mul_fixed(rg.g_tab, xr), te_mul_glv(input, xr), ad, ad_len, out192, pk, blinding_raw, tr);
    pedersen_begin_blind(pk, te_mul_fixed(rg.b_tab, blinding_raw), out192, blinded, tr);
}
// Second half: nonces, R, Ok, challenge, responses.  Writes R | Ok | s | sb into out192 + 64.
template <class S>
DR_HD_COLD void pedersen_prove_finish(const S& rg, const uint8_t* sk32, const TEAffine& input, const uint32_t* blinding_raw, const VrfHash& tr, uint8_t* out192) {
    Fn x = fp_from_le_bytes_mod<Fn>(sk32, 32);
    Fn b = Fn::zero();
    for (int i = 0; i < 8; i++) b.v[i] = blinding_raw[i];
    b = b.to_mont();
    uint32_t kr[8], kbr[8];
    Fn k = vrf_nonce(tr, x);
    Fn kb = vrf_nonce(tr, b);
    fn_raw_limbs(kr, k);
    fn_raw_limbs(kbr, kb);
    TEAffine R, ok;
    te_to_affine2(te_add(te_mul_fixed(rg.g_tab, kr), te_mul_fixed(rg.b_tab, kbr)), te_mul_glv(input, kr), R, ok);
    VrfHash tc = tr;
    tc.update_byte(0x40);
    sha_absorb_point(tc, R);
    sha_absorb_point(tc, ok);
    uint8_t cb[16];
    vrf_squeeze(tc, cb, 16);
    Fn c = fp_from_le_bytes_mod<Fn>(cb, 16);
    Fn s = k + c * x;
    Fn sb = kb + c * b;
    te_encode(out192 + 64, R);
    te_encode(out192 + 96, ok);
    fn_to_le_bytes(out192 + 128, s);
    fn_to_le_bytes(out192 + 160, sb);
}
// Writes O | Ybar | R | Ok | s | sb; returns the public key, the blinded key and the blinding factor.
template <class S>
DR_HD_COLD void pedersen_prove_core(const S& rg, const uint8_t* sk32, const uint8_t* msg, uint32_t msg_len, const uint8_t* ad, uint32_t ad_len, uint8_t* out192,
                                    TEAffine& pk, TEAffine& blinded, uint32_t* blinding_raw) {
    TEAffine input = vrf_encode_to_curve(rg, msg, msg_len);
    VrfHash tr;
    pedersen_prove_begin(rg, sk32, input, ad, ad_len, out192, pk, blinded, blinding_raw, tr);
    pedersen_prove_finish(rg, sk32, input, blinding_raw, tr, out192);
}

// Window table for te_mul_fixed: thread (w, c) of 32 x 16 writes the 16 entries d = 16c .. 16c + 15 of window w.
struct TeFixedTableBody {
    DR_HD void operator()(const BlockCtx& ctx, TEAffine base, TEPre* out) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < (uint32_t)TE_FIXED_WINDOWS * 16) {
                const uint32_t w = i >> 4, first = (i & 15) * 16;
                TEExt step = TEExt::from_affine(base);
#pragma unroll 1
                for (uint32_t j = 0; j < 8 * w; j++) step = te_dbl(step);
                TEExt cur = TEExt::identity();
#pragma unroll 1
                for (int bit = 7; bit >= 0; bit--) {
                    cur = te_dbl(cur);
                    if ((first >> bit) & 1) cur = te_add(cur, step);
                }
#pragma unroll 1
                for (uint32_t d = first; d < first + 16; d++) {
                    out[256 * w + d] = TEPre::from_affine(d ? te_to_affine(cur) : TEAffine::identity());
                    cur = te_add(cur, step);
                }
            }
        }
    }
};

// First half of the Pedersen prover, eight threads per proof (te_coop.cuh).  This kernel is on the critical path of a pass whatever
// its width, so its serial chains are spread over the lanes: the two Elligator 2 maps of hash-to-curve (a field inversion and a
// square root each) run side by side, sk * H(alpha) is a cooperative variable-base multiplication, sk * G and b * B are split by
// table windows.  What remains on one lane: the affine conversions, the SHA-512 / SHAKE transcripts and the point encodings.
DR_HD size_t pedersen_start_smem(uint32_t threads) { return (threads / COOP_LANES) * (sizeof(TeCoopState) + 2 * sizeof(TEAffine)); }
struct PedersenStartBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const RingTab* tab, const ProveInput* in, const uint8_t* blob, ProofState* st, uint32_t count) const {
        const uint32_t items = ctx.nthreads / COOP_LANES;
        TeCoopState* cs = (TeCoopState*)ctx.smem;
        TEAffine* maps = (TEAffine*)(cs + items);  // [items][2]
        // A. hash-to-curve maps on lanes 0 and 1
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            if (lane == 0) cs[item].live = p < count ? 1u : 0u;
            if (p < count && lane < 2) {
                const ProveInput& pi = in[p];
                uint8_t u[96];
                h2c_uniform_bytes(rg, blob + pi.alpha_off, pi.alpha_len, u);
                maps[2 * item + lane] = te_map_to_curve_ell2(fr_from_be48_mod(u + 48 * lane));
            }
        }
        DR_BLOCK_SYNC();
        // B. input point = 4 * (map(u0) + map(u1))  (te_affine_point.py:213-222); operands of sk * input
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            if (p < count && lane == 0) {
                TeCoopState& s = cs[item];
                TEExt sum = te_add(TEExt::from_affine(maps[2 * item]), TEExt::from_affine(maps[2 * item + 1]));
                const TEAffine input = te_to_affine(te_dbl(te_dbl(sum)));
                st[p].vrf_input = input;
                // sk * input = k1 * (+-input) + k2 * (+-psi(input)) with 128-bit halves (te.cuh te_glv_split): half the doublings
                uint32_t xr[8];
                fn_raw_limbs(xr, fp_from_le_bytes_mod<Fn>(in[p].sk, 32));
                bool n1, n2;
                te_glv_split(xr, s.k, n1, s.k2, n2);
                coop_set_point(s.tab[0], TEExt::from_affine(n1 ? te_neg(input) : input));
                const TEExt psi = te_endomorphism(input);
                coop_set_point(s.tab2[0], n2 ? te_neg(psi) : psi);
            }
        }
        DR_BLOCK_SYNC();
        te_straus_coop(ctx, cs, 4, 4);
        // C. sk * G by windows
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, p = ctx.bx * items + item;
            TeCoopState& s = cs[item];
            if (s.live) {
                uint32_t xr[8];
                fn_raw_limbs(xr, fp_from_le_bytes_mod<Fn>(in[p].sk, 32));
                te_mul_fixed_coop_partial(t % COOP_LANES, rg.g_tab, xr, s.part);
            }
        }
        DR_BLOCK_SYNC();
        // D. public key, output point, transcript, blinding factor (one lane); the public key waits in s.m for step F
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            if (p < count && lane == 0) {
                TeCoopState& s = cs[item];
                ProofState& ps = st[p];
                const ProveInput& pi = in[p];
                const TEExt output{s.acc.c[CX], s.acc.c[CY], s.acc.c[CZ], s.acc.c[CT]};
                TEAffine pk;
                pedersen_begin_transcript(rg, fp_from_le_bytes_mod<Fn>(pi.sk, 32), ps.vrf_input, te_fold_fixed_coop(s.part), output, blob + pi.ad_off, pi.ad_len, ps.pedersen,
                                          pk, ps.t, ps.vrf_tr);
                s.m[0] = pk.x;
                s.m[1] = pk.y;
                for (int i = 0; i < 8; i++) s.k[i] = ps.t[i];
            }
        }
        DR_BLOCK_SYNC();
        // E. b * B by windows
        DR_THREAD_LOOP(t, ctx) {
            TeCoopState& s = cs[t / COOP_LANES];
            if (s.live) te_mul_fixed_coop_partial(t % COOP_LANES, rg.b_tab, s.k, s.part);
        }
        DR_BLOCK_SYNC();
        // F. blinded key; ring-membership check of the producer key against the item's ring
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            const uint32_t ring = p < count ? in[p].ring : 0u;
            const TEAffine* nm = tab[ring].nm;
            const uint32_t max_ring = tab[ring].max_ring;
            if (p < count && lane == 0) {
                TeCoopState& s = cs[item];
                ProofState& ps = st[p];
                const ProveInput& pi = in[p];
                const TEAffine pk{s.m[0], s.m[1]};
                TEAffine blinded;
                pedersen_begin_blind(pk, te_fold_fixed_coop(s.part), ps.pedersen, blinded, ps.vrf_tr);
                ps.k = pi.k;
                ps.ring = ring;
                ps.relation = blinded;
                // producer_key must be pk(sk) and sit at row k of the ring (vrf/ring/vrf.py:196-197, members.py:71-81)
                ps.status = (pi.k < max_ring && nm[pi.k] == pk) ? 0u : 1u;
            }
        }
    }
};
// The start of a bare ring proof (RingProofBuilder.build, proof_builder.py:38-69) from a caller's blinding factor t, in place of
// PedersenStartBody: relation = PK_k + t * B, with t * B split by table windows over eight lanes per proof as in step E above.  No
// hash-to-curve, no sk * G, no Pedersen transcript; the host has checked t < order and k < max_ring.
DR_HD size_t ring_proof_start_smem(uint32_t threads) { return (size_t)threads * sizeof(TEExt); }
struct RingProofStartBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const RingTab* tab, const ProveInput* in, ProofState* st, uint32_t count) const {
        const uint32_t items = ctx.nthreads / COOP_LANES;
        TEExt* part = (TEExt*)ctx.smem;  // [items][COOP_LANES]
        auto limbs = [](uint32_t* out, const uint8_t* le32) {
            for (int i = 0; i < 8; i++)
                out[i] = (uint32_t)le32[4 * i] | (uint32_t)le32[4 * i + 1] << 8 | (uint32_t)le32[4 * i + 2] << 16 | (uint32_t)le32[4 * i + 3] << 24;
        };
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, p = ctx.bx * items + item;
            if (p < count) {
                uint32_t tr[8];
                limbs(tr, in[p].sk);
                te_mul_fixed_coop_partial(t % COOP_LANES, rg.b_tab, tr, part + COOP_LANES * item);
            }
        }
        DR_BLOCK_SYNC();
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            const uint32_t ring = p < count ? in[p].ring : 0u;
            const TEAffine* nm = tab[ring].nm;
            if (p < count && lane == 0) {
                ProofState& ps = st[p];
                const ProveInput& pi = in[p];
                ps.k = pi.k;
                ps.ring = ring;
                limbs(ps.t, pi.sk);
                ps.relation = te_to_affine(te_add(TEExt::from_affine(nm[pi.k]), te_fold_fixed_coop(part + COOP_LANES * item)));
                ps.status = 0;
            }
        }
    }
};

// Second half, one thread per proof; nothing of the ring proof depends on it, so it runs on the side stream.
struct PedersenFinishBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const ProveInput* in, ProofState* st, uint32_t count) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t p = ctx.bx * ctx.nthreads + t;
            if (p < count) {
                ProofState& ps = st[p];
                pedersen_prove_finish(rg, in[p].sk, ps.vrf_input, ps.t, ps.vrf_tr, ps.pedersen);
            }
        }
    }
};

// ---- B. witness accumulators (columns.py:127-146), 32 threads per proof ------------------------------------
// acc_0 = seed; the only rows that change it are row k (adds PK_k) and the 253 bit rows (add 2^j * B when bit j of the blinding
// factor is set).  The 253 running sums are a prefix scan over group elements: lane l owns bit rows 8l .. 8l+7, sums them,
// the lane totals are scanned in five rounds through shared memory, and each lane then walks its rows from its offset.  The affine
// values the reference computes with one inversion per addition come from one inversion per lane (Montgomery's trick over the
// lane's rows; the 32 inversions of a proof run side by side).
constexpr uint32_t WIT_LANES = 32, WIT_ROWS = 8;
static_assert(WIT_LANES * WIT_ROWS >= SCALAR_BITS, "every bit row needs a lane");
DR_HD size_t witness_coop_smem(uint32_t threads) { return (size_t)2 * threads * sizeof(TEExt); }
struct WitnessBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const RingTab* tab, ProofState* st, uint32_t count) const {
        TEExt* sm = (TEExt*)ctx.smem;  // two scan buffers of nthreads entries
        const uint32_t T = ctx.nthreads, ppb = T / WIT_LANES;
        auto bit_of = [](const ProofState& ps, uint32_t j) { return (ps.t[j >> 5] >> (j & 31)) & 1u; };
        // the proof's ring, resolved per warp (one proof per warp) before any branch on lane data
        auto ring_of = [&](uint32_t p) -> const RingTab& { return tab[p < count ? st[p].ring : 0u]; };
        // 1. lane totals (lane 0 starts from a0 = seed + PK_k)
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t lane = t % WIT_LANES, p = ctx.bx * ppb + t / WIT_LANES;
            const RingTab& rt = ring_of(p);
            const TEAffine* nm = rt.nm;
            const uint32_t max_ring = rt.max_ring;
            TEExt acc = TEExt::identity();
            if (p < count) {
                const ProofState& ps = st[p];
                if (lane == 0) acc = te_add(TEExt::from_affine(rg.seed), TEExt::from_affine(nm[ps.k < max_ring ? ps.k : 0]));
#pragma unroll 1
                for (uint32_t j = lane * WIT_ROWS; j < (lane + 1) * WIT_ROWS && j < SCALAR_BITS; j++)
                    if (bit_of(ps, j)) acc = te_add(acc, TEExt::from_affine(nm[max_ring + j]));
            }
            sm[t] = acc;
        }
        DR_BLOCK_SYNC();
        // 2. inclusive scan over the lanes of every proof (ping-pong between the two buffers)
        uint32_t cur = 0;
        for (uint32_t d = 1; d < WIT_LANES; d <<= 1) {
            DR_THREAD_LOOP(t, ctx) {
                const uint32_t lane = t % WIT_LANES;
                TEExt a = sm[cur * T + t];
                if (lane >= d) a = te_add(a, sm[cur * T + t - d]);
                sm[(cur ^ 1) * T + t] = a;
            }
            DR_BLOCK_SYNC();
            cur ^= 1;
        }
        // 3. walk the lane's rows from the sum of everything before them; affine through one inversion per lane
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t lane = t % WIT_LANES, p = ctx.bx * ppb + t / WIT_LANES;
            const RingTab& rt = ring_of(p);
            const TEAffine* nm = rt.nm;
            const uint32_t max_ring = rt.max_ring;
            if (p < count) {
                ProofState& ps = st[p];
                const TEExt a0 = te_add(TEExt::from_affine(rg.seed), TEExt::from_affine(nm[ps.k < max_ring ? ps.k : 0]));
                TEExt acc = lane ? sm[cur * T + t - 1] : a0;
                Fr zs[WIT_ROWS], pre[WIT_ROWS];
                Fr run = lane ? Fr::one() : a0.Z;
                uint32_t rows = 0;
#pragma unroll 1
                for (uint32_t j = lane * WIT_ROWS; j < (lane + 1) * WIT_ROWS && j < SCALAR_BITS; j++, rows++) {
                    if (bit_of(ps, j)) acc = te_add(acc, TEExt::from_affine(nm[max_ring + j]));
                    ps.s[j] = {acc.X, acc.Y};  // projective for now
                    zs[rows] = acc.Z;
                    pre[rows] = run;
                    run = run * acc.Z;
                }
                Fr inv_run = run.inv();
#pragma unroll 1
                for (uint32_t i = rows; i-- > 0;) {
                    const uint32_t j = lane * WIT_ROWS + i;
                    Fr zi = inv_run * pre[i];
                    inv_run = inv_run * zs[i];
                    ps.s[j] = {ps.s[j].x * zi, ps.s[j].y * zi};
                }
                if (lane == 0) ps.a0 = {a0.X * inv_run, a0.Y * inv_run};  // inv_run == 1 / Z_a0
            }
        }
        DR_BLOCK_SYNC();
        // 4. consistency check and transcript start, one lane per proof
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t lane = t % WIT_LANES, p = ctx.bx * ppb + t / WIT_LANES;
            const Shake128* prefix = ring_of(p).prefix;
            if (p < count && lane == 0) {
                ProofState& ps = st[p];
                // the accumulator must end at seed + relation (proof_builder.py:66-69)
                TEExt chk = te_add(TEExt::from_affine(rg.seed), TEExt::from_affine(ps.relation));
                if (!te_ext_eq_affine(chk, ps.s[SCALAR_BITS - 1])) ps.status |= 2u;
                // transcript: copy the ring prefix, absorb the instance (phases.py:18-26)
                Shake128 tr = *prefix;
                shake_absorb_label(tr, "instance", 8);
                shake_absorb_fr(tr, ps.relation.x);
                shake_absorb_fr(tr, ps.relation.y);
                tr.absorb_be32(64);
                ps.tr = tr;
            }
        }
    }
};

// Column synthesis (columns.py:111-146 + 43-53): value of witness column `col` at row `row`.  `max_ring` is the proof's ring's
// (RingTab::max_ring), which the caller resolves once per block.
DR_HD Fr witness_eval(const RingDev& rg, uint32_t max_ring, const ProofState& ps, uint32_t col, uint32_t row) {
    const uint32_t N = rg.N;
    if (row >= N - 3) return ps.zk[3 * col + (row - (N - 3))];
    if (col == COL_B) {
        if (row < max_ring) return row == ps.k ? Fr::one() : Fr::zero();
        uint32_t j = row - max_ring;
        if (j < SCALAR_BITS && ((ps.t[j >> 5] >> (j & 31)) & 1)) return Fr::one();
        return Fr::zero();
    }
    if (col == COL_ACCIP) return row > ps.k ? Fr::one() : Fr::zero();
    const TEAffine* pt;
    if (row <= ps.k)
        pt = &rg.seed;
    else if (row <= max_ring)
        pt = &ps.a0;
    else {
        // max_ring_size below the domain's capacity leaves more than 253 blinding-base rows (members.py:46-51); the b column
        // is zero there (columns.py:111-124), so the accumulator keeps its final value
        uint32_t j = row - max_ring - 1;
        pt = &ps.s[j < SCALAR_BITS ? j : SCALAR_BITS - 1];
    }
    return col == COL_ACCX ? pt->x : pt->y;
}

// ---- C. witness interpolation: grid (4 columns, proofs) ------------------------------------------------
struct WitnessInttBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const RingTab* tab, const ProofState* st, Fr* wit_coef) const {
        const ProofState& ps = st[ctx.by];
        const uint32_t max_ring = tab[ps.ring].max_ring;
        uint32_t col = ctx.bx;
        Fr* dst = wit_coef + ((size_t)ctx.by * 4 + col) * rg.N;
        Fr ninv = rg.n_inv;
        ntt_block(
            ctx, rg.N, rg.logN, rg.tw_inv, [&](uint32_t r) { return witness_eval(rg, max_ring, ps, col, r); }, [&](uint32_t k, const Fr& v) { dst[k] = v * ninv; });
    }
};

// ---- D'. witness commitments from the evaluation form: grid (4 columns, proofs) ---------------------------------
// A witness column is piecewise constant (b: one-hot + bits, acc_ip: a step, acc_x / acc_y: change only where a bit
// of the blinding factor is set) except for its three blinding rows, so in the Lagrange basis
//   C = sum_i v_i [L_i(tau)]_1 = sum_{j=1..N} (v_{j-1} - v_j) S_j,   S_j = sum_{i<j} [L_i(tau)]_1,  v_N := 0
// has ~130 non-zero terms instead of N.  It is the same group element as KZG.commit(interpolate(v))
// (columns.py:29-60), hence the same bytes; the S_j have their own fixed-base window table per ring.
// Two phases per (column, proof) block: (1) the threads scan the rows and compact the non-zero steps, with their signed
// window digits, into shared memory; (2) the (step, window) pairs are dealt round-robin to the threads, so every lane
// issues the same number of table additions however the steps are distributed over the rows.
constexpr uint32_t WC_MAX_STEPS = 272;  // <= 1 (row k) + 253 (bit rows) + 3 blinding rows + slack, per column
// shared memory: [steps: WC_MAX_STEPS x (row, flip, W digits) as int16] [rows found: WC_MAX_STEPS x int16]
// [unit steps: WC_MAX_STEPS x (row, negate) as int16] [3 counters] [per-thread partial sums]
DR_HD size_t witness_commit_steps_bytes(uint32_t W) { return (((size_t)WC_MAX_STEPS * (2 + W + 1 + 2) * sizeof(int16_t) + 16 + 15) / 16) * 16; }
DR_HD size_t witness_commit_smem(uint32_t W, uint32_t threads) { return witness_commit_steps_bytes(W) + threads * sizeof(G1); }
struct WitnessCommitBody {
    DR_HD void operator()(const BlockCtx& ctx, const G1Affine* table, TableGeom g, RingDev rg, const RingTab* tab, const ProofState* st, G1* out) const {
        int16_t* steps = (int16_t*)ctx.smem;
        const uint32_t stride = 2 + g.W;
        int16_t* rows = steps + (size_t)WC_MAX_STEPS * stride;
        int16_t* units = rows + WC_MAX_STEPS;
        uint32_t* counters = (uint32_t*)(units + 2 * WC_MAX_STEPS);  // rows found, full steps, unit steps
        G1* sm = (G1*)(ctx.smem + witness_commit_steps_bytes(g.W));
        const ProofState& ps = st[ctx.by];
        const uint32_t max_ring = tab[ps.ring].max_ring;
        const uint32_t col = ctx.bx, N = rg.N;
        DR_THREAD_LOOP(t, ctx) {
            if (t < 3) counters[t] = 0;
        }
        DR_BLOCK_SYNC();
        // 1a. find the rows where the column steps (cheap, every lane busy)
        DR_THREAD_LOOP(t, ctx) {
#pragma unroll 1
            for (uint32_t j = 1 + t; j <= N; j += ctx.nthreads) {
                Fr d = witness_eval(rg, max_ring, ps, col, j - 1);
                if (j < N) d = d - witness_eval(rg, max_ring, ps, col, j);
                if (d.is_zero()) continue;
                uint32_t slot = atomic_add_u32(&counters[0], 1u);
                if (slot < WC_MAX_STEPS) rows[slot] = (int16_t)j;  // base S_j is table point j - 1 (N <= 4096)
            }
        }
        DR_BLOCK_SYNC();
        // 1b. one step per lane.  Steps of +-1 (the b column, acc_ip) are one table entry each and go to their own list, so
        // that phase 2 does not walk W windows of zero digits for them; the others get their W signed digits.
        const uint32_t found = counters[0] < WC_MAX_STEPS ? counters[0] : WC_MAX_STEPS;
        DR_THREAD_LOOP(t, ctx) {
#pragma unroll 1
            for (uint32_t slot = t; slot < found; slot += ctx.nthreads) {
                const uint32_t j = (uint32_t)(uint16_t)rows[slot];
                Fr d = witness_eval(rg, max_ring, ps, col, j - 1);
                if (j < N) d = d - witness_eval(rg, max_ring, ps, col, j);
                Fr kc = d.from_mont(), nk = d.neg().from_mont();
                bool flip = (nk.v[1] | nk.v[2] | nk.v[3] | nk.v[4] | nk.v[5] | nk.v[6] | nk.v[7]) == 0;  // use the shorter of d, -d
                if (flip) kc = nk;
                if (kc.v[0] == 1 && (kc.v[1] | kc.v[2] | kc.v[3] | kc.v[4] | kc.v[5] | kc.v[6] | kc.v[7]) == 0) {
                    uint32_t u = atomic_add_u32(&counters[2], 1u);
                    units[2 * u] = (int16_t)j;
                    units[2 * u + 1] = flip ? 1 : 0;
                    continue;
                }
                int16_t* s = steps + (size_t)atomic_add_u32(&counters[1], 1u) * stride;
                s[0] = (int16_t)j;
                s[1] = flip ? 1 : 0;
                uint32_t carry = 0;
#pragma unroll 1
                for (uint32_t w = 0; w < g.W; w++) s[2 + w] = (int16_t)msm_digit(kc.v, w, g, carry);
            }
        }
        DR_BLOCK_SYNC();
        // 2. (step, window) pairs and unit steps dealt round-robin to the lanes
        const uint32_t full = counters[1] * g.W, total = full + counters[2];
        DR_THREAD_LOOP(t, ctx) {
            G1 acc = G1::inf();
            // the entry of the next pair is fetched before the current addition is issued
            int dg = 0;
            bool neg = false;
            G1Affine pt = G1Affine::inf();
            auto fetch = [&](uint32_t it, int& dg_o, bool& neg_o, G1Affine& pt_o) {
                if (it < full) {
                    const int16_t* s = steps + (size_t)(it / g.W) * stride;
                    const uint32_t w = it % g.W;
                    dg_o = s[2 + w];
                    neg_o = (dg_o < 0) != (s[1] != 0);
                    if (dg_o) pt_o = table[g.entry((uint32_t)(uint16_t)s[0] - 1u, w, (uint32_t)(dg_o < 0 ? -dg_o : dg_o))];
                } else {
                    const int16_t* u = units + 2 * (size_t)(it - full);
                    dg_o = 1;
                    neg_o = u[1] != 0;
                    pt_o = table[g.entry((uint32_t)(uint16_t)u[0] - 1u, 0, 1u)];
                }
            };
            if (t < total) fetch(t, dg, neg, pt);
#pragma unroll 1
            for (uint32_t it = t; it < total; it += ctx.nthreads) {
                const uint32_t nx = it + ctx.nthreads;
                int dg_next = 0;
                bool neg_next = false;
                G1Affine pt_next = pt;
                if (nx < total) fetch(nx, dg_next, neg_next, pt_next);
                if (dg) g1_madd(acc, pt, neg);
                dg = dg_next;
                neg = neg_next;
                pt = pt_next;
            }
            sm[t] = acc;
        }
        DR_BLOCK_SYNC();
        for (uint32_t stride2 = ctx.nthreads >> 1; stride2 > 0; stride2 >>= 1) {
            DR_STRIDE_LOOP(t, stride2, ctx) {
                G1 a = sm[t];
                g1_add(a, sm[t + stride2]);
                sm[t] = a;
            }
            DR_BLOCK_SYNC();
        }
        DR_THREAD_LOOP(t, ctx) {
            if (t == 0) out[(size_t)ctx.by * 4 + col] = sm[0];
        }
    }
};

// ---- E. transcript phase 1: committed columns -> 7 alphas (phases.py:18-26) ------------------------------
struct Transcript1Body {
    DR_HD void operator()(const BlockCtx& ctx, ProofState* st, uint32_t count) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t p = ctx.bx * ctx.nthreads + t;
            if (p < count) {
                ProofState& ps = st[p];
                Shake128 tr = ps.tr;  // absorb byte by byte into a local copy, not into HBM
                shake_absorb_label(tr, "committed_cols", 14);
                for (int i = 0; i < 4; i++) shake_absorb_g1(tr, ps.commits[i]);
                tr.absorb_be32(4 * 96);
                Fr alpha[7];
                shake_challenges(tr, "constraints_aggregation", 23, alpha, 7);
                for (int i = 0; i < 7; i++) ps.alpha[i] = alpha[i];
                ps.tr = tr;
            }
        }
    }
};

// ---- F. 4x low-degree extension of the witness columns: grid (16 = 4 cosets x 4 columns, proofs) ---------
struct WitnessLdeBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const RingTab* tab, const ProofState* st, const Fr* wit_coef, Fr* lde) const {
        uint32_t col = ctx.bx & 3, j = ctx.bx >> 2;
        const Fr* src = wit_coef + ((size_t)ctx.by * 4 + col) * rg.N;
        Fr* dst = lde + (((size_t)ctx.by * 4 + col) * 4 + j) * rg.N;
        const uint32_t mask = 4 * rg.N - 1;
        if (j == 0) {  // coset 0 is the N-domain itself: the column's own evaluations, no transform needed
            const ProofState& ps = st[ctx.by];
            const uint32_t max_ring = tab[ps.ring].max_ring;
            DR_STRIDE_LOOP(i, rg.N, ctx) { dst[i] = witness_eval(rg, max_ring, ps, col, i); }
            return;
        }
        ntt_block(
            ctx, rg.N, rg.logN, rg.tw_fwd, [&](uint32_t k) { return j ? src[k] * rg.w4[(j * k) & mask] : src[k]; }, [&](uint32_t i, const Fr& v) { dst[i] = v; });
    }
};

// Plain coset LDE of `count` coefficient vectors (ring set-up: px, py, s, L_0, L_last): grid (4*count)
struct PlainLdeBody {
    DR_HD void operator()(const BlockCtx& ctx, uint32_t N, uint32_t logN, const Fr* tw_fwd, const Fr* w4, const Fr* coef, Fr* lde) const {
        uint32_t v = ctx.bx >> 2, j = ctx.bx & 3;
        const Fr* src = coef + (size_t)v * N;
        Fr* dst = lde + ((size_t)v * 4 + j) * N;
        const uint32_t mask = 4 * N - 1;
        ntt_block(
            ctx, N, logN, tw_fwd, [&](uint32_t k) { return j ? src[k] * w4[(j * k) & mask] : src[k]; }, [&](uint32_t i, const Fr& val) { dst[i] = val; });
    }
};

// ---- large domains (N > 4096, outside the reference: params.py:172-173 rejects them) -----------------------------------
// The transform no longer fits one CTA, so the fused loaders / storers above become element-wise passes around the
// two-pass NTT of ntt.cuh: materialise the witness evaluations, pre-twist the cosets, untwist after the inverse transform.
struct WitnessEvalBody {  // grid (ceil(N / threads), 4 columns, proofs): out[(p*4 + col)*N + r] = column value at row r
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const RingTab* tab, const ProofState* st, Fr* out) const {
        const ProofState& ps = st[ctx.bz];
        const uint32_t max_ring = tab[ps.ring].max_ring;
        DR_THREAD_LOOP(t, ctx) {
            uint32_t r = ctx.bx * ctx.nthreads + t;
            if (r < rg.N) out[((size_t)ctx.bz * 4 + ctx.by) * rg.N + r] = witness_eval(rg, max_ring, ps, ctx.by, r);
        }
    }
};
struct CosetTwistBody {  // grid (ceil(N / threads), 4 cosets, vectors): out[(v*4 + j)*N + k] = in[v*N + k] * w4^(j k)
    DR_HD void operator()(const BlockCtx& ctx, uint32_t N, const Fr* w4, const Fr* in, Fr* out) const {
        const uint32_t j = ctx.by, mask = 4 * N - 1;
        DR_THREAD_LOOP(t, ctx) {
            uint32_t k = ctx.bx * ctx.nthreads + t;
            if (k < N) {
                Fr x = in[(size_t)ctx.bz * N + k];
                out[((size_t)ctx.bz * 4 + j) * N + k] = j ? x * w4[((uint64_t)j * k) & mask] : x;
            }
        }
    }
};
struct CosetUntwistBody {  // grid (ceil(N / threads), 4 cosets, vectors): buf[(v*4 + j)*N + k] *= w4^(-j k)
    DR_HD void operator()(const BlockCtx& ctx, uint32_t N, const Fr* w4inv, Fr* buf) const {
        const uint32_t j = ctx.by, mask = 4 * N - 1;
        DR_THREAD_LOOP(t, ctx) {
            uint32_t k = ctx.bx * ctx.nthreads + t;
            if (k < N && j) {
                Fr* e = buf + ((size_t)ctx.bz * 4 + j) * N + k;
                *e = *e * w4inv[((uint64_t)j * k) & mask];
            }
        }
    }
};

// ---- G. constraints c1..c7 and their alpha-aggregation on the 4N domain (constraints.py:64-151,
//         proof_builder.py:165-179): grid (ceil(4N / threads), proofs) ----------------------------------------
struct ConstraintBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const RingTab* tab, const ProofState* st, const Fr* lde, Fr* agg) const {
        const ProofState& ps = st[ctx.by];
        const uint32_t N = rg.N, N4 = 4 * rg.N;
        const Fr* w = lde + (size_t)ctx.by * 4 * N4;
        const Fr *b4 = w + COL_B * N4, *ax4 = w + COL_ACCX * N4, *ay4 = w + COL_ACCY * N4, *aip4 = w + COL_ACCIP * N4;
        const Fr* fl = tab[ps.ring].fixed_lde;
        const Fr *px4 = fl, *py4 = fl + N4, *s4 = fl + 2 * N4, *l0 = fl + 3 * N4, *ln = fl + 4 * N4, *nl = fl + 5 * N4;
        Fr* out = agg + (size_t)ctx.by * N4;
        const TEAffine rps = ps.s[SCALAR_BITS - 1];  // result + seed
        DR_THREAD_LOOP(t, ctx) {
            uint32_t p = ctx.bx * ctx.nthreads + t;
            if (p < N4) {
                uint32_t j = p / N, i = p - j * N;
                if (j == 0 && i + 3 < N) {
                    // coset 0 is the N-domain itself: every constraint holds on rows 0 .. N-4 (that is what the quotient's
                    // divisibility by X^N - 1 expresses), only the three blinding rows contribute
                    out[p] = Fr::zero();
                    continue;
                }
                uint32_t q = j * N + ((i + 1) & (N - 1));  // row shifted by 4 in the 4N domain
                Fr one = Fr::one();
                Fr x1 = ax4[p], y1 = ay4[p], x2 = px4[p], y2 = py4[p], x3 = ax4[q], y3 = ay4[q];
                Fr bi = b4[p], nli = nl[p], aip = aip4[p];
                Fr omb = one - bi;
                Fr x1y1 = x1 * y1, y2x2 = y2 * x2;
                Fr c1 = (aip4[q] - aip - bi * s4[p]) * nli;
                Fr xt = x3 * (y1 * y2 - fr_mul5(x1 * x2)) - (x1y1 + y2x2);
                Fr c2 = (bi * xt + omb * (x3 - x1)) * nli;
                Fr yt = y3 * (x1 * y2 - x2 * y1) - (x1y1 - y2x2);
                Fr c3 = (bi * yt + omb * (y3 - y1)) * nli;
                Fr c4 = bi * omb;
                Fr l0i = l0[p], lni = ln[p];
                Fr c5 = (x1 - rg.seed.x) * l0i + (x1 - rps.x) * lni;
                Fr c6 = (y1 - rg.seed.y) * l0i + (y1 - rps.y) * lni;
                Fr c7 = aip * l0i + (aip - one) * lni;
                out[p] = c1 * ps.alpha[0] + c2 * ps.alpha[1] + c3 * ps.alpha[2] + c4 * ps.alpha[3] + c5 * ps.alpha[4] + c6 * ps.alpha[5] + c7 * ps.alpha[6];
            }
        }
    }
};

// ---- H. inverse transform of the aggregated constraint, coset by coset: grid (4, proofs) ------------------
// After this kernel agg[j*N + k0] holds  w4^(-j*k0) * (1/N) * sum_i E[4i+j] w^(-i*k0).
struct QuotientInttBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, Fr* agg) const {
        uint32_t j = ctx.bx;
        Fr* buf = agg + ((size_t)ctx.by * 4 + j) * rg.N;
        const uint32_t mask = 4 * rg.N - 1;
        Fr ninv = rg.n_inv;
        ntt_block(
            ctx, rg.N, rg.logN, rg.tw_inv, [&](uint32_t i) { return buf[i]; },
            [&](uint32_t k0, const Fr& v) {
                Fr r = v * ninv;
                buf[k0] = j ? r * rg.w4inv[(j * k0) & mask] : r;
            });
    }
};

// ---- I. 4-point combine across cosets -> coefficients c[0..4N) of the aggregated polynomial ---------------
// c[k0 + N*m] = 1/4 * sum_j i4^(-j*m) * D_j[k0],  i4 = w4^N (primitive 4th root of unity).
struct QuotientCombineBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const Fr* agg, Fr* cagg) const {
        const uint32_t N = rg.N;
        const Fr* src = agg + (size_t)ctx.by * 4 * N;
        Fr* dst = cagg + (size_t)ctx.by * 4 * N;
        DR_THREAD_LOOP(t, ctx) {
            uint32_t k0 = ctx.bx * ctx.nthreads + t;
            if (k0 < N) {
                Fr d0 = src[k0], d1 = src[N + k0], d2 = src[2 * N + k0], d3 = src[3 * N + k0];
                Fr i4inv = rg.w4inv[N];  // i4^-1
                Fr s02 = d0 + d2, m02 = d0 - d2, s13 = d1 + d3, m13 = (d1 - d3) * i4inv;
                // m = 0: d0+d1+d2+d3 ; m = 1: d0 + i^-1 d1 - d2 - i^-1 d3 ; m = 2: d0-d1+d2-d3 ; m = 3: d0 - i^-1 d1 - d2 + i^-1 d3
                dst[k0] = (s02 + s13) * rg.quarter;
                dst[N + k0] = (m02 + m13) * rg.quarter;
                dst[2 * N + k0] = (s02 - s13) * rg.quarter;
                dst[3 * N + k0] = (m02 - m13) * rg.quarter;
            }
        }
    }
};

// ---- J. multiply by the tail-vanishing cubic and divide by X^N - 1 (proof_builder.py:181-195,
//         ops.py:207-224): q[j] = sum_{i>=1, iN+j<=4N+3} e[iN+j],  e = c * tail.  grid (ceil((3N+1)/threads), proofs)
struct QuotientFoldBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const Fr* cagg, Fr* quot, uint32_t qstride) const {
        const uint32_t N = rg.N, N4 = 4 * rg.N;
        const Fr* c = cagg + (size_t)ctx.by * N4;
        Fr* q = quot + (size_t)ctx.by * qstride;
        DR_THREAD_LOOP(t, ctx) {
            uint32_t j = ctx.bx * ctx.nthreads + t;
            if (j < qstride) {
                // e[idx] = sum_{tt=0..3} tail[tt] * c[idx - tt], q[j] = sum_idx e[idx]: sum the taps first, multiply once per tap
                // (tail[3] = 1): 3 multiplications per coefficient instead of up to 16
                Fr taps[4] = {Fr::zero(), Fr::zero(), Fr::zero(), Fr::zero()};
                for (uint32_t idx = N + j; idx < N4 + 4; idx += N) {
#pragma unroll
                    for (uint32_t tt = 0; tt < 4; tt++) {
                        if (idx >= tt && idx - tt < N4) taps[tt] = taps[tt] + c[idx - tt];
                    }
                }
                q[j] = rg.tail[0] * taps[0] + rg.tail[1] * taps[1] + rg.tail[2] * taps[2] + taps[3];
            }
        }
    }
};

// ---- transcript phase 2: quotient commitment -> zeta (phases.py:29-32) ---------------------------------------
struct Transcript2Body {
    DR_HD void operator()(const BlockCtx& ctx, ProofState* st, uint32_t count) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t p = ctx.bx * ctx.nthreads + t;
            if (p < count) {
                ProofState& ps = st[p];
                Shake128 tr = ps.tr;
                shake_absorb_label(tr, "quotient", 8);
                shake_absorb_g1(tr, ps.commits[4]);
                tr.absorb_be32(96);
                Fr zeta;
                shake_challenges(tr, "evaluation_point", 16, &zeta, 1);
                ps.zeta = zeta;
                ps.tr = tr;
            }
        }
    }
};

// Parallel Horner: value of poly (n coefficients, n a multiple of nthreads or padded by the caller) at x.
// All threads of the block cooperate; result valid for every thread after the call (read from smem[0]).
DR_HD Fr block_poly_eval(const BlockCtx& ctx, const Fr* poly, uint32_t n, const Fr& x, Fr* sm) {
    const uint32_t T = ctx.nthreads;
    const uint32_t L = (n + T - 1) / T;
    DR_THREAD_LOOP(t, ctx) {
        uint32_t lo = t * L, hi = lo + L < n ? lo + L : n;
        Fr acc = Fr::zero();
        if (lo < n) {
#pragma unroll 1
            for (uint32_t k = hi; k > lo; k--) acc = acc * x + poly[k - 1];
            // times x^lo
            Fr pw = Fr::one(), base = x;
            uint32_t e = lo;
#pragma unroll 1
            while (e) {
                if (e & 1) pw = pw * base;
                base = base.sqr();
                e >>= 1;
            }
            acc = acc * pw;
        }
        sm[t] = acc;
    }
    DR_BLOCK_SYNC();
    for (uint32_t stride = T >> 1; stride > 0; stride >>= 1) {
        DR_STRIDE_LOOP(t, stride, ctx) { sm[t] = sm[t] + sm[t + stride]; }
        DR_BLOCK_SYNC();
    }
    Fr r = sm[0];
    DR_BLOCK_SYNC();
    return r;
}

// ---- K. evaluations at zeta (proof_builder.py:243-267): grid (7, proofs) ----------------------------------------
// slot order = payload order: px, py, s, b, accip, accx, accy
struct EvalBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const RingTab* tab, ProofState* st, const Fr* wit_coef) const {
        ProofState& ps = st[ctx.by];
        uint32_t slot = ctx.bx;
        const Fr* poly;
        const Fr* wc = wit_coef + (size_t)ctx.by * 4 * rg.N;
        const Fr* fc = tab[ps.ring].fixed_coef;
        switch (slot) {
            case 0: poly = fc; break;
            case 1: poly = fc + rg.N; break;
            case 2: poly = fc + 2 * rg.N; break;
            case 3: poly = wc + COL_B * rg.N; break;
            case 4: poly = wc + COL_ACCIP * rg.N; break;
            case 5: poly = wc + COL_ACCX * rg.N; break;
            default: poly = wc + COL_ACCY * rg.N; break;
        }
        Fr v = block_poly_eval(ctx, poly, rg.N, ps.zeta, (Fr*)ctx.smem);
        DR_THREAD_LOOP(t, ctx) {
            if (t == 0) ps.evals[slot] = v;
        }
    }
};

// ---- linearisation polynomial (proof_builder.py:197-241): grid (ceil(N/threads), proofs) --------------------------
DR_HD void lin_factors(const RingDev& rg, const ProofState& ps, Fr& f_ip, Fr& f_x, Fr& f_y) {
    Fr one = Fr::one();
    Fr st = ps.zeta - rg.w_last;
    Fr b = ps.evals[3], x1 = ps.evals[5], y1 = ps.evals[6], x2 = ps.evals[0], y2 = ps.evals[1];
    Fr omb = one - b;
    Fr fx = (b * (y1 * y2 - fr_mul5(x1 * x2)) + omb) * st;
    Fr fy = (b * (x1 * y2 - x2 * y1) + omb) * st;
    f_ip = st * ps.alpha[0];
    f_x = fx * ps.alpha[1];
    f_y = fy * ps.alpha[2];
}
struct LinPolyBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const ProofState* st, const Fr* wit_coef, Fr* lin) const {
        const ProofState& ps = st[ctx.by];
        const Fr* wc = wit_coef + (size_t)ctx.by * 4 * rg.N;
        Fr* dst = lin + (size_t)ctx.by * rg.N;
        Fr f_ip, f_x, f_y;
        lin_factors(rg, ps, f_ip, f_x, f_y);
        DR_THREAD_LOOP(t, ctx) {
            uint32_t k = ctx.bx * ctx.nthreads + t;
            if (k < rg.N) dst[k] = wc[COL_ACCIP * rg.N + k] * f_ip + wc[COL_ACCX * rg.N + k] * f_x + wc[COL_ACCY * rg.N + k] * f_y;
        }
    }
};
// L(zeta * w): grid (1, proofs)
struct LinEvalBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, ProofState* st, const Fr* lin) const {
        ProofState& ps = st[ctx.by];
        Fr zw = ps.zeta * rg.omega;
        Fr v = block_poly_eval(ctx, lin + (size_t)ctx.by * rg.N, rg.N, zw, (Fr*)ctx.smem);
        DR_THREAD_LOOP(t, ctx) {
            if (t == 0) ps.lzw = v;
        }
    }
};

// ---- transcript phase 3 (phases.py:35-43) -------------------------------------------------------------------------
struct Transcript3Body {
    DR_HD void operator()(const BlockCtx& ctx, ProofState* st, uint32_t count) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t p = ctx.bx * ctx.nthreads + t;
            if (p < count) {
                ProofState& ps = st[p];
                Shake128 tr = ps.tr;
                shake_absorb_label(tr, "register_evaluations", 20);
                for (int i = 0; i < 7; i++) shake_absorb_fr(tr, ps.evals[i]);
                tr.absorb_be32(7 * 32);
                shake_absorb_label(tr, "shifted_linearization_evaluation", 32);
                shake_absorb_fr(tr, ps.lzw);
                tr.absorb_be32(32);
                Fr nu[8];
                shake_challenges(tr, "kzg_aggregation", 15, nu, 8);
                for (int i = 0; i < 8; i++) ps.nu[i] = nu[i];
                ps.tr = tr;
            }
        }
    }
};

// ---- M. aggregated opening polynomial (proof_builder.py:288-315): grid (ceil((3N+1)/threads), proofs) ------------
struct AggOpenBody {
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const RingTab* tab, const ProofState* st, const Fr* wit_coef, const Fr* quot, uint32_t qstride,
                          Fr* aggopen) const {
        const ProofState& ps = st[ctx.by];
        const Fr* fc = tab[ps.ring].fixed_coef;
        const uint32_t N = rg.N;
        const Fr* wc = wit_coef + (size_t)ctx.by * 4 * N;
        const Fr* q = quot + (size_t)ctx.by * qstride;
        Fr* dst = aggopen + (size_t)ctx.by * qstride;
        DR_THREAD_LOOP(t, ctx) {
            uint32_t k = ctx.bx * ctx.nthreads + t;
            if (k < 3 * N + 1) {
                Fr acc = q[k] * ps.nu[7];
                if (k < N) {
                    acc = acc + fc[k] * ps.nu[0] + fc[N + k] * ps.nu[1] + fc[2 * N + k] * ps.nu[2] +
                          wc[COL_B * N + k] * ps.nu[3] + wc[COL_ACCIP * N + k] * ps.nu[4] + wc[COL_ACCX * N + k] * ps.nu[5] + wc[COL_ACCY * N + k] * ps.nu[6];
                }
                dst[k] = acc;
            }
        }
    }
};

// ---- N. synthetic division by (X - x) (pcs/utils.py:27-35): in place, poly[i] <- q[i], one block per polynomial.
// r_i = sum_{k>=i} a_k x^(k-i);  q_i = r_{i+1}, q_{n-1} = 0.
DR_HD size_t synthetic_div_smem(uint32_t threads) { return ((size_t)5 * threads + 1) * sizeof(Fr); }
DR_HD void block_synthetic_div(const BlockCtx& ctx, Fr* poly, uint32_t n, const Fr& x, Fr* sm) {
    const uint32_t T = ctx.nthreads;
    const uint32_t L = (n + T - 1) / T;
    // pass 1: suffix sums local to each chunk, written in place
    DR_THREAD_LOOP(t, ctx) {
        uint32_t lo = t * L, hi = lo + L < n ? lo + L : n;
        Fr acc = Fr::zero();
        if (lo < n) {
#pragma unroll 1
            for (uint32_t k = hi; k > lo; k--) {
                acc = acc * x + poly[k - 1];
                poly[k - 1] = acc;
            }
        }
        sm[t] = acc;  // local suffix at the chunk start
    }
    DR_BLOCK_SYNC();
    // pass 2: full suffix at each chunk start, R_t = S_t + x^(len_t) * R_{t+1}: a suffix scan of affine maps.  Every chunk holds
    // (A_t, B_t) with R_t = A_t + B_t * R_{t+d}; a round composes it with the pair d chunks further on, so log2(T) rounds of two
    // multiplications replace a serial walk over all chunks by one thread (which was most of this kernel's time).
    // sm layout: [0, T] S / final carries (pass 4 reads entry T), then two ping-pong pairs of T entries each: 5 T + 1 elements
    Fr* A0 = sm + T + 1;
    Fr* B0 = A0 + T;
    Fr* A1 = B0 + T;
    Fr* B1 = A1 + T;
    const uint32_t nchunks = (n + L - 1) / L;
    DR_THREAD_LOOP(t, ctx) {
        if (t < nchunks) {
            const uint32_t len = (t + 1) * L <= n ? L : n - t * L;
            Fr mult = Fr::one(), base = x;
            uint32_t e = len;
#pragma unroll 1
            while (e) {
                if (e & 1) mult = mult * base;
                base = base.sqr();
                e >>= 1;
            }
            A0[t] = sm[t];
            B0[t] = mult;
        }
    }
    DR_BLOCK_SYNC();
    bool flip = false;
    for (uint32_t d = 1; d < nchunks; d <<= 1) {
        Fr *Ai = flip ? A1 : A0, *Bi = flip ? B1 : B0, *Ao = flip ? A0 : A1, *Bo = flip ? B0 : B1;
        DR_THREAD_LOOP(t, ctx) {
            if (t < nchunks) {
                if (t + d < nchunks) {
                    Ao[t] = Ai[t] + Bi[t] * Ai[t + d];
                    Bo[t] = Bi[t] * Bi[t + d];
                } else {  // nothing beyond: R_{t+d} = 0
                    Ao[t] = Ai[t];
                    Bo[t] = Bi[t];
                }
            }
        }
        DR_BLOCK_SYNC();
        flip = !flip;
    }
    {
        const Fr* R = flip ? A1 : A0;  // R[t] = full suffix at the start of chunk t
        DR_THREAD_LOOP(t, ctx) {
            if (t < nchunks) sm[t] = t + 1 < nchunks ? R[t + 1] : Fr::zero();  // what chunk t needs: R_{t+1}
        }
    }
    DR_BLOCK_SYNC();
    // pass 3: r_i = local_i + x^(hi - i) * R_{t+1}
    DR_THREAD_LOOP(t, ctx) {
        uint32_t lo = t * L, hi = lo + L < n ? lo + L : n;
        if (lo < n) {
            Fr carry = sm[t];
            Fr pw = x;  // x^(hi - (hi-1))
#pragma unroll 1
            for (uint32_t k = hi; k > lo; k--) {
                poly[k - 1] = poly[k - 1] + pw * carry;
                pw = pw * x;
            }
        }
    }
    DR_BLOCK_SYNC();
    // pass 4: shift down by one: q_i = r_{i+1}.  Chunk boundaries need the neighbour's first element.
    DR_THREAD_LOOP(t, ctx) {
        uint32_t lo = t * L;
        sm[t] = lo < n ? poly[lo] : Fr::zero();  // r at chunk start
    }
    DR_BLOCK_SYNC();
    DR_THREAD_LOOP(t, ctx) {
        uint32_t lo = t * L, hi = lo + L < n ? lo + L : n;
        if (lo < n) {
            for (uint32_t k = lo; k + 1 < hi; k++) poly[k] = poly[k + 1];
            poly[hi - 1] = (hi < n) ? sm[t + 1] : Fr::zero();
        }
    }
    DR_BLOCK_SYNC();
}
struct OpenQuotientsBody {
    // grid (2, proofs): bx = 0 -> aggregated poly at zeta (3N+1 coefficients), bx = 1 -> L at zeta*w (N)
    DR_HD void operator()(const BlockCtx& ctx, RingDev rg, const ProofState* st, Fr* aggopen, uint32_t qstride, Fr* lin) const {
        const ProofState& ps = st[ctx.by];
        if (ctx.bx == 0) {
            block_synthetic_div(ctx, aggopen + (size_t)ctx.by * qstride, 3 * rg.N + 1, ps.zeta, (Fr*)ctx.smem);
        } else {
            Fr zw = ps.zeta * rg.omega;
            block_synthetic_div(ctx, lin + (size_t)ctx.by * rg.N, rg.N, zw, (Fr*)ctx.smem);
        }
    }
};

// ---- P. proof assembly (vrf/ring/vrf.py:51-58, proof_payload.py:68-91): 784 bytes per proof ----------------------
// the 592-byte ring-proof payload (proof_payload.py:68-91)
DR_HD void encode_ring_payload(uint8_t* o, const ProofState& ps) {
    for (int i = 0; i < 4; i++) g1_compress(o + 48 * i, ps.commits[i]);
    o += 192;
    for (int i = 0; i < 7; i++) fr_to_le_bytes_raw(o + 32 * i, ps.evals[i].from_mont());
    o += 224;
    g1_compress(o, ps.commits[4]);
    fr_to_le_bytes_raw(o + 48, ps.lzw.from_mont());
    g1_compress(o + 80, ps.commits[5]);
    g1_compress(o + 128, ps.commits[6]);
}
struct FinalizeBody {
    DR_HD void operator()(const BlockCtx& ctx, const ProofState* st, uint32_t count, uint8_t* out, uint32_t* status) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t p = ctx.bx * ctx.nthreads + t;
            if (p < count) {
                const ProofState& ps = st[p];
                uint8_t* o = out + 784 * (size_t)p;
                for (int i = 0; i < 192; i++) o[i] = ps.pedersen[i];
                encode_ring_payload(o + 192, ps);
                status[p] = ps.status;
            }
        }
    }
};
// Bare ring proofs: relations (x | y, 32-byte little-endian each) at out[64 p ..), payloads at out[64 count + 592 p ..).  The
// blinding factor is the last thing of the proof state that identifies the signer (relation - t * B = PK_k): it is cleared here.
struct RingProofFinalizeBody {
    DR_HD void operator()(const BlockCtx& ctx, ProofState* st, uint32_t count, uint8_t* out) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t p = ctx.bx * ctx.nthreads + t;
            if (p < count) {
                ProofState& ps = st[p];
                fr_to_le_bytes_raw(out + 64 * (size_t)p, ps.relation.x.from_mont());
                fr_to_le_bytes_raw(out + 64 * (size_t)p + 32, ps.relation.y.from_mont());
                encode_ring_payload(out + 64 * (size_t)count + 592 * (size_t)p, ps);
                for (int i = 0; i < 8; i++) ps.t[i] = 0;
            }
        }
    }
};

// scatter commit results (one per proof) into ProofState::commits[slot]
struct StoreCommitBody {
    // slot for result c of a proof = byte c of `slot_map`
    DR_HD void operator()(const BlockCtx& ctx, const G1Affine* res, uint32_t per_proof, uint32_t slot_map, ProofState* st, uint32_t count) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t idx = ctx.bx * ctx.nthreads + t;
            if (idx < count * per_proof) {
                uint32_t p = idx / per_proof, c = idx % per_proof;
                st[p].commits[(slot_map >> (8 * c)) & 0xff] = res[idx];
            }
        }
    }
};

// blinding rows: n x 12 canonical 32-byte values -> Montgomery in ProofState::zk (null -> zeros)
struct ZkRowsBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* raw, ProofState* st, uint32_t count) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t idx = ctx.bx * ctx.nthreads + t;
            if (idx < count * 12) {
                Fr v = Fr::zero();
                if (raw) {
                    fr_from_le_bytes_raw(v, raw + 32 * (size_t)idx);
                    while (!v.is_canonical_raw()) Fr::sub_mod_inplace(v.v);
                    v = v.to_mont();
                }
                st[idx / 12].zk[idx % 12] = v;
            }
        }
    }
};

// ---- ring set-up helpers ----------------------------------------------------------------------------------------
// The public-vector row of one 32-byte key: undecodable / identity / out-of-subgroup keys become the padding point
// (members.py:36-41,61-69).
DR_HD TEAffine ring_key_point(const uint8_t* key, const TEAffine& padding) {
    TEAffine p;
    if (!te_decode_checked(p, key)) p = padding;
    return p;
}
// keys (32 bytes each) -> nm[i]
struct KeyDecodeBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* keys, uint32_t n_keys, TEAffine padding, TEAffine* nm) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < n_keys) nm[i] = ring_key_point(keys + 32 * (size_t)i, padding);
        }
    }
};
// Evaluations of the fixed columns of several rings at once (dr_ring_roots_from_keys): block row k < n_rings writes ring k's px and
// py at out[2kN ..) and out[(2k+1)N ..), row i being its key key_off[k] + i while i < key_off[k+1] - key_off[k] and the
// key-independent row tail[i] (padding, 2^j B, zeros) after that; block row n_rings, when launched, writes the selector s
// (i < max_ring) at out[2 n_rings N ..).
struct RingRootColumnsBody {
    DR_HD void operator()(const BlockCtx& ctx, const TEAffine* tail, const uint8_t* keys, const uint32_t* key_off, uint32_t n_rings, uint32_t N, uint32_t max_ring,
                          TEAffine padding, Fr* out) const {
        const uint32_t k = ctx.by;
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < N) {
                if (k == n_rings) {
                    out[2 * (size_t)n_rings * N + i] = i < max_ring ? Fr::one() : Fr::zero();
                } else {
                    const uint32_t first = key_off[k], count = key_off[k + 1] - first;
                    const TEAffine p = i < count ? ring_key_point(keys + 32 * ((size_t)first + i), padding) : tail[i];
                    out[2 * (size_t)k * N + i] = p.x;
                    out[(2 * (size_t)k + 1) * N + i] = p.y;
                }
            }
        }
    }
};
// Change of the px / py evaluations when row rows[j] goes from old_keys[j] (null: the padding point) to new_keys[j], keys mapped as in
// ring_key_point: out[rows[j]] = dx, out[N + rows[j]] = dy; the other rows of out stay as they are (zero).  Rows are distinct.
struct RootDeltaBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* old_keys, const uint8_t* new_keys, const uint32_t* rows, uint32_t n, uint32_t N, TEAffine padding,
                          Fr* out) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t j = ctx.bx * ctx.nthreads + t;
            if (j < n) {
                const TEAffine from = old_keys ? ring_key_point(old_keys + 32 * (size_t)j, padding) : padding;
                const TEAffine to = ring_key_point(new_keys + 32 * (size_t)j, padding);
                out[rows[j]] = to.x - from.x;
                out[N + rows[j]] = to.y - from.y;
            }
        }
    }
};
// column evaluations for the fixed columns: out[0][i] = nm[i].x, out[1][i] = nm[i].y, out[2][i] = i < max_ring
struct FixedColumnsBody {
    DR_HD void operator()(const BlockCtx& ctx, const TEAffine* nm, uint32_t N, uint32_t max_ring, Fr* out) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < N) {
                out[i] = nm[i].x;
                out[N + i] = nm[i].y;
                out[2 * N + i] = i < max_ring ? Fr::one() : Fr::zero();
            }
        }
    }
};
// notlast[j*N + i] = w4^(4i + j) - w^(N-4)
struct NotLastBody {
    DR_HD void operator()(const BlockCtx& ctx, uint32_t N, const Fr* w4, Fr w_last, Fr* out) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t p = ctx.bx * ctx.nthreads + t;
            if (p < 4 * N) {
                uint32_t j = p / N, i = p - j * N;
                out[p] = w4[4 * i + j] - w_last;
            }
        }
    }
};

}  // namespace dr
