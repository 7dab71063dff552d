// Verification kernels (batched): Tiny / Pedersen VRF verification and the ring-proof verifier.
//
// Device restatement of
//   dot_ring/vrf/ietf/tiny.py:72-83                     TinyVRF.verify
//   dot_ring/vrf/pedersen/vrf.py:48-73,128-143          PedersenVRF.decode / verify
//   dot_ring/vrf/primitives.py:85-144                   challenge, vrf_transcript, delinearisation
//   dot_ring/ring_proof/proof_payload.py:93-143         payload decode (lengths, canonical scalars, G1 validity)
//   dot_ring/ring_proof/transcript/phases.py:46-69      derive_challenges_after_vk
//   dot_ring/ring_proof/verify.py:51-210                quotient / linearisation terms, two LinearPcsVerifications
//   dot_ring/ring_proof/pcs/kzg.py:56-108,304-338       random-linear-combined KZG check, 2 Miller loops + final exp
// Work is split so that every launch has (items x sub-tasks) threads: point decodes (sqrt + subgroup check) are one thread per
// (item, point), G1 scalar multiplications one per (item, term, GLV half), the Bandersnatch equations of the VRF schemes run on
// eight cooperating lanes per item (te_coop.cuh), ring transcripts / scalar algebra on one thread per item, the pairing on a warp.  Verdict codes: 1 valid, 0 invalid, 2 malformed (where the reference raises ValueError).
#pragma once
#include "pairing.cuh"
#include "pairing_warp.cuh"
#include "ring.cuh"

namespace dr {

struct SuiteDev {  // VRF suite constants (dot_ring/curve/specs/bandersnatch.py:48-107)
    TEAffine generator, blinding_base;
    const TEPre* g_tab;  // te_mul_fixed tables of the generator / blinding base (provers and the Pedersen verifier)
    const TEPre* b_tab;
    uint32_t suite_id_len;
    uint8_t suite_id[32];
    uint32_t dst_len;
    uint8_t dst[64];
    uint32_t hash_kind;  // 0 SHA-512, 1 SHAKE128 (ring.cuh: VrfHash)
};

struct VerifyInput {  // host-packed per item: salt|alpha and ad inside the blob
    uint32_t in_off, in_len, ad_off, ad_len;
};

constexpr uint32_t ST_MALFORMED = 1, ST_PEDERSEN_BAD = 2;

DR_HD void load_le_limbs8(uint32_t* out, const uint8_t* in, int nbytes) {
    for (int i = 0; i < 8; i++) out[i] = 0;
    for (int b = 0; b < nbytes; b++) out[b >> 2] |= (uint32_t)in[b] << (8 * (b & 3));
}

// ---- decode + subgroup check, one thread per point (vrf/codec.py:39-45) ------------------------------------
// in: count encodings of 32 bytes at in + stride*(i / per_item) + 32*(i % per_item)
struct TeDecodeManyBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* in, uint32_t stride, uint32_t per_item, uint32_t count, TEAffine* out, uint8_t* ok) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < count) {
                TEAffine p;
                bool good = te_decode_checked(p, in + (size_t)stride * (i / per_item) + 32 * (i % per_item));
                out[i] = good ? p : TEAffine::identity();
                ok[i] = good ? 1 : 0;
            }
        }
    }
};

// Pedersen verification equations for one decoded proof; pts = O, Ybar, R, Ok.  Returns status bits.
template <class S>
DR_HD_COLD uint32_t pedersen_verify_core(const S& su, const TEAffine* pts, const uint8_t* ok4, const uint8_t* proof192, const uint8_t* msg, uint32_t msg_len,
                                         const uint8_t* ad, uint32_t ad_len) {
    if (!(ok4[0] && ok4[1] && ok4[2] && ok4[3])) return ST_MALFORMED;
    uint32_t ks[3][8];
    load_le_limbs8(ks[0], proof192 + 128, 32);  // s
    load_le_limbs8(ks[1], proof192 + 160, 32);  // sb
    if (Fn::geq_mod(ks[0]) || Fn::geq_mod(ks[1])) return ST_MALFORMED;
    TEAffine input = vrf_encode_to_curve(su, msg, msg_len);
    VrfHash tr;
    tr.init(su.hash_kind);
    tr.update(su.suite_id, su.suite_id_len);
    tr.update_byte(0x02);
    uint8_t le[8] = {1, 0, 0, 0, 0, 0, 0, 0};
    tr.update(le, 8);
    sha_absorb_point(tr, input);
    sha_absorb_point(tr, pts[0]);
    for (int i = 0; i < 8; i++) le[i] = i < 4 ? (uint8_t)(ad_len >> (8 * i)) : 0;
    tr.update(le, 8);
    tr.update(ad, ad_len);
    sha_absorb_point(tr, pts[1]);
    tr.update_byte(0x40);
    sha_absorb_point(tr, pts[2]);
    sha_absorb_point(tr, pts[3]);
    uint8_t cb[16];
    vrf_squeeze(tr, cb, 16);
    uint32_t c[8];
    load_le_limbs8(c, cb, 16);
    // s*I - c*O == Ok: s split by the endomorphism, one 32-window Straus pass over (I, psi(I), -O)
    bool ok = te_ext_eq_affine(te_glv_straus2(input, ks[0], TEExt::from_affine(te_neg(pts[0])), c), pts[3]);
    // s*G + sb*B - c*Ybar == R: the two fixed bases from their window tables (no doublings), the blinded key by a 128-bit multiplication
    const TEAffine nyb = te_neg(pts[1]);
    TEExt lhs = te_add(te_mul_fixed(su.g_tab, ks[0]), te_mul_fixed(su.b_tab, ks[1]));
    lhs = te_add(lhs, te_mul_raw(nyb, c, 4));
    ok = ok && te_ext_eq_affine(lhs, pts[2]);
    return ok ? 0u : ST_PEDERSEN_BAD;
}

// One thread per proof (large batches: every lane of a warp busy with its own item, throughput-bound); pts / ok hold the 4 decoded
// points of every proof.  Small batches use the eight-lane kernels below (latency-bound).
struct PedersenVerifySerialBody {
    DR_HD void operator()(const BlockCtx& ctx, SuiteDev su, const VerifyInput* in, const uint8_t* blob, const uint8_t* proofs, uint32_t proof_stride, const TEAffine* pts,
                          const uint8_t* ok, uint32_t count, uint32_t* status) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < count) {
                const VerifyInput& vi = in[i];
                status[i] = pedersen_verify_core(su, pts + 4 * (size_t)i, ok + 4 * (size_t)i, proofs + (size_t)proof_stride * i, blob + vi.in_off, vi.in_len, blob + vi.ad_off,
                                                 vi.ad_len);
            }
        }
    }
};

// Tiny (ietf/tiny.py:72-83) and Thin (ietf/thin.py:84-99) verification, one thread per item (large batches).  Both schemes share the
// transcript over the two I/O pairs (G, PK), (I, O) and the delinearised pair (G + z I, PK + z O); they differ in the
// scheme byte and in what the proof carries:  tiny  O (32) | c (16) | s (32): recompute R, compare the challenge;
//                                              thin  O (32) | R (32) | s (32): derive c from R, check s I' - c O' == R.
// pts = decoded points per item: [O, PK] (tiny) or [O, R, PK] (thin).  status bit0 malformed, bit1 invalid.
struct IetfVerifySerialBody {
    DR_HD void operator()(const BlockCtx& ctx, SuiteDev su, uint32_t thin, const VerifyInput* in, const uint8_t* blob, const uint8_t* proofs, const TEAffine* pts,
                          const uint8_t* ok, uint32_t count, uint32_t* status) const {
        const uint32_t npts = thin ? 3 : 2, plen = thin ? 96 : 80;
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < count) {
                const VerifyInput& vi = in[i];
                const uint8_t* pr = proofs + (size_t)plen * i;
                uint32_t st = 0;
                uint32_t ks[2][8];
                load_le_limbs8(ks[0], pr + (thin ? 64 : 48), 32);  // s
                bool decoded = true;
                for (uint32_t j = 0; j < npts; j++) decoded = decoded && ok[(size_t)npts * i + j];
                if (!decoded || Fn::geq_mod(ks[0])) st = ST_MALFORMED;
                if (!st) {
                    const TEAffine out = pts[(size_t)npts * i], pk = pts[(size_t)npts * i + npts - 1];
                    TEAffine input = vrf_encode_to_curve(su, blob + vi.in_off, vi.in_len);
                    VrfHash tr;
                    tr.init(su.hash_kind);
                    tr.update(su.suite_id, su.suite_id_len);
                    tr.update_byte(thin ? 0x01 : 0x00);
                    uint8_t le[8] = {2, 0, 0, 0, 0, 0, 0, 0};
                    tr.update(le, 8);
                    sha_absorb_point(tr, su.generator);
                    sha_absorb_point(tr, pk);
                    sha_absorb_point(tr, input);
                    sha_absorb_point(tr, out);
                    for (int b = 0; b < 8; b++) le[b] = b < 4 ? (uint8_t)(vi.ad_len >> (8 * b)) : 0;
                    tr.update(le, 8);
                    tr.update(blob + vi.ad_off, vi.ad_len);
                    // delinearisation scalar z (primitives.py:128-144), merged pair (G + z I, PK + z O)
                    VrfHash td = tr;
                    td.update_byte(0x30);
                    uint8_t zb[16];
                    vrf_squeeze(td, zb, 16);
                    uint32_t z[8];
                    load_le_limbs8(z, zb, 16);
                    // R = s*I' - c*O' with I' = G + z I, O' = PK + z O, expanded: s*G + (s z)*I - c*PK - (c z)*O.  s*G comes from the
                    // generator's window table; the rest is ONE 32-window Straus pass over (I, psi(I), -O, psi(-O), -PK) with the
                    // two full-length scalars split by the endomorphism -- instead of two 128-bit multiplications, two affine
                    // conversions and a second pass.
                    tr.update_byte(0x40);
                    if (thin) {
                        sha_absorb_point(tr, pts[(size_t)npts * i + 1]);
                        uint8_t cb[16];
                        vrf_squeeze(tr, cb, 16);
                        load_le_limbs8(ks[1], cb, 16);
                    } else {
                        load_le_limbs8(ks[1], pr + 32, 16);  // c
                    }
                    auto fn_of = [](const uint32_t* limbs) {
                        Fn v;
                        for (int l = 0; l < 8; l++) v.v[l] = limbs[l];
                        return v.to_mont();
                    };
                    const Fn zf = fn_of(z);
                    uint32_t sz[8], cz[8];
                    fn_raw_limbs(sz, fn_of(ks[0]) * zf);
                    fn_raw_limbs(cz, fn_of(ks[1]) * zf);
                    TEExt res = te_glv_straus3(input, sz, te_neg(out), cz, TEExt::from_affine(te_neg(pk)), ks[1]);
                    res = te_add(res, te_mul_fixed(su.g_tab, ks[0]));
                    if (thin) {
                        if (!te_ext_eq_affine(res, pts[(size_t)npts * i + 1])) st = ST_PEDERSEN_BAD;
                    } else {
                        sha_absorb_point(tr, te_to_affine(res));
                        uint8_t cb[16];
                        vrf_squeeze(tr, cb, 16);
                        bool same = true;
                        for (int b = 0; b < 16; b++) same = same && (cb[b] == pr[32 + b]);
                        if (!same) st = ST_PEDERSEN_BAD;
                    }
                }
                status[i] = st;
            }
        }
    }
};

// Pedersen verification, eight threads per proof (te_coop.cuh); pts / ok hold the 4 decoded points of every proof.
// One thread per proof ran ~7 k dependent field multiplications (7 ms whatever the batch size, 255 registers, 12 % occupancy); here
// the Elligator maps take two lanes, s*I - c*O is a cooperative two-point Straus, c*Ybar a cooperative 128-bit multiplication and
// s*G + sb*B come from the fixed-base window tables, split by windows over the lanes.
DR_HD size_t vrf_verify_coop_smem(uint32_t threads) { return (threads / COOP_LANES) * (sizeof(TeCoopState) + 2 * sizeof(TEAffine) + 16); }
struct PedersenVerifyBody {
    DR_HD void operator()(const BlockCtx& ctx, SuiteDev su, const VerifyInput* in, const uint8_t* blob, const uint8_t* proofs, uint32_t proof_stride, const TEAffine* pts,
                          const uint8_t* ok, uint32_t count, uint32_t* status) const {
        const uint32_t items = ctx.nthreads / COOP_LANES;
        TeCoopState* cs = (TeCoopState*)ctx.smem;
        TEAffine* maps = (TEAffine*)(cs + items);             // [items][2]
        uint32_t* good = (uint32_t*)(maps + 2 * items);        // [items]: first equation holds
        auto malformed = [&](uint32_t p) {
            const uint8_t* o = ok + 4 * (size_t)p;
            uint32_t ks[8], kb[8];
            load_le_limbs8(ks, proofs + (size_t)proof_stride * p + 128, 32);
            load_le_limbs8(kb, proofs + (size_t)proof_stride * p + 160, 32);
            return !(o[0] && o[1] && o[2] && o[3]) || Fn::geq_mod(ks) || Fn::geq_mod(kb);
        };
        // A. decode status; hash-to-curve maps on lanes 0 and 1
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            const bool bad = p < count && malformed(p);
            if (lane == 0) {
                cs[item].live = p < count && !bad ? 1u : 0u;
                if (p < count) status[p] = bad ? ST_MALFORMED : 0u;
            }
            if (p < count && !bad && lane < 2) {
                const VerifyInput& vi = in[p];
                uint8_t u[96];
                h2c_uniform_bytes(su, blob + vi.in_off, vi.in_len, u);
                maps[2 * item + lane] = te_map_to_curve_ell2(fr_from_be48_mod(u + 48 * lane));
            }
        }
        DR_BLOCK_SYNC();
        // B. input point, transcript, challenge; operands of s*I - c*O
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            TeCoopState& s = cs[item];
            if (s.live && lane == 0) {
                const VerifyInput& vi = in[p];
                const TEAffine* pt = pts + 4 * (size_t)p;  // O, Ybar, R, Ok
                const uint8_t* pr = proofs + (size_t)proof_stride * p;
                TEExt sum = te_add(TEExt::from_affine(maps[2 * item]), TEExt::from_affine(maps[2 * item + 1]));
                const TEAffine input = te_to_affine(te_dbl(te_dbl(sum)));
                VrfHash tr;
                tr.init(su.hash_kind);
                tr.update(su.suite_id, su.suite_id_len);
                tr.update_byte(0x02);
                uint8_t le[8] = {1, 0, 0, 0, 0, 0, 0, 0};
                tr.update(le, 8);
                sha_absorb_point(tr, input);
                sha_absorb_point(tr, pt[0]);
                for (int i = 0; i < 8; i++) le[i] = i < 4 ? (uint8_t)(vi.ad_len >> (8 * i)) : 0;
                tr.update(le, 8);
                tr.update(blob + vi.ad_off, vi.ad_len);
                sha_absorb_point(tr, pt[1]);
                tr.update_byte(0x40);
                sha_absorb_point(tr, pt[2]);
                sha_absorb_point(tr, pt[3]);
                uint8_t cb[16];
                vrf_squeeze(tr, cb, 16);
                coop_set_point(s.tab[0], TEExt::from_affine(input));
                coop_set_point(s.tab2[0], TEExt::from_affine(te_neg(pt[0])));
                load_le_limbs8(s.k, pr + 128, 32);  // s
                load_le_limbs8(s.k2, cb, 16);       // c
            }
        }
        DR_BLOCK_SYNC();
        te_straus_coop(ctx, cs, 8, 4);
        // C. s*I - c*O == Ok ?  then the operand of -c*Ybar
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            TeCoopState& s = cs[item];
            if (s.live && lane == 0) {
                const TEAffine* pt = pts + 4 * (size_t)p;
                good[item] = te_ext_eq_affine(coop_get_point(s.acc), pt[3]) ? 1u : 0u;
                coop_set_point(s.tab[0], TEExt::from_affine(te_neg(pt[1])));
                for (int i = 0; i < 8; i++) s.k[i] = s.k2[i];
            }
        }
        DR_BLOCK_SYNC();
        te_straus_coop(ctx, cs, 4, 0);
        // D. s*G by table windows; E. fold it, sb*B by table windows; F. s*G + sb*B - c*Ybar == R ?
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            TeCoopState& s = cs[item];
            if (s.live) {
                uint32_t ks[8];
                load_le_limbs8(ks, proofs + (size_t)proof_stride * p + 128, 32);
                te_mul_fixed_coop_partial(lane, su.g_tab, ks, s.part);
            }
        }
        DR_BLOCK_SYNC();
        DR_THREAD_LOOP(t, ctx) {
            TeCoopState& s = cs[t / COOP_LANES];
            if (s.live && t % COOP_LANES == 0) coop_set_point(s.acc, te_add(coop_get_point(s.acc), te_fold_fixed_coop(s.part)));
        }
        DR_BLOCK_SYNC();
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            TeCoopState& s = cs[item];
            if (s.live) {
                uint32_t kb[8];
                load_le_limbs8(kb, proofs + (size_t)proof_stride * p + 160, 32);
                te_mul_fixed_coop_partial(lane, su.b_tab, kb, s.part);
            }
        }
        DR_BLOCK_SYNC();
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            TeCoopState& s = cs[item];
            if (s.live && lane == 0) {
                const TEAffine* pt = pts + 4 * (size_t)p;
                const TEExt total = te_add(coop_get_point(s.acc), te_fold_fixed_coop(s.part));
                status[p] = (good[item] && te_ext_eq_affine(total, pt[2])) ? 0u : ST_PEDERSEN_BAD;
            }
        }
    }
};

// Tiny (ietf/tiny.py:72-83) and Thin (ietf/thin.py:84-99) verification, eight threads per item.  Both schemes share the
// transcript over the two I/O pairs (G, PK), (I, O) and the delinearised pair (G + z I, PK + z O); they differ in the
// scheme byte and in what the proof carries:  tiny  O (32) | c (16) | s (32): recompute R, compare the challenge;
//                                              thin  O (32) | R (32) | s (32): derive c from R, check s I' - c O' == R.
// pts = decoded points per item: [O, PK] (tiny) or [O, R, PK] (thin).  status bit0 malformed, bit1 invalid.
// z*I and z*O are cooperative 128-bit multiplications, s*I' - c*O' a cooperative two-point Straus (te_coop.cuh).
struct IetfVerifyBody {
    DR_HD void operator()(const BlockCtx& ctx, SuiteDev su, uint32_t thin, const VerifyInput* in, const uint8_t* blob, const uint8_t* proofs, const TEAffine* pts,
                          const uint8_t* ok, uint32_t count, uint32_t* status) const {
        const uint32_t npts = thin ? 3 : 2, plen = thin ? 96 : 80;
        const uint32_t items = ctx.nthreads / COOP_LANES;
        TeCoopState* cs = (TeCoopState*)ctx.smem;
        TEAffine* maps = (TEAffine*)(cs + items);  // [items][2]; after step B: maps[2 item] = the input point
        auto malformed = [&](uint32_t p) {
            uint32_t ks[8];
            load_le_limbs8(ks, proofs + (size_t)plen * p + (thin ? 64 : 48), 32);  // s
            bool decoded = true;
            for (uint32_t j = 0; j < npts; j++) decoded = decoded && ok[(size_t)npts * p + j];
            return !decoded || Fn::geq_mod(ks);
        };
        // A. decode status; hash-to-curve maps on lanes 0 and 1
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            const bool bad = p < count && malformed(p);
            if (lane == 0) {
                cs[item].live = p < count && !bad ? 1u : 0u;
                if (p < count) status[p] = bad ? ST_MALFORMED : 0u;
            }
            if (p < count && !bad && lane < 2) {
                const VerifyInput& vi = in[p];
                uint8_t u[96];
                h2c_uniform_bytes(su, blob + vi.in_off, vi.in_len, u);
                maps[2 * item + lane] = te_map_to_curve_ell2(fr_from_be48_mod(u + 48 * lane));
            }
        }
        DR_BLOCK_SYNC();
        // transcript up to the additional data (shared by steps B and E)
        auto transcript = [&](uint32_t p, const TEAffine& input, VrfHash& tr) {
            const VerifyInput& vi = in[p];
            tr.init(su.hash_kind);
            tr.update(su.suite_id, su.suite_id_len);
            tr.update_byte(thin ? 0x01 : 0x00);
            uint8_t le[8] = {2, 0, 0, 0, 0, 0, 0, 0};
            tr.update(le, 8);
            sha_absorb_point(tr, su.generator);
            sha_absorb_point(tr, pts[(size_t)npts * p + npts - 1]);
            sha_absorb_point(tr, input);
            sha_absorb_point(tr, pts[(size_t)npts * p]);
            for (int b = 0; b < 8; b++) le[b] = b < 4 ? (uint8_t)(vi.ad_len >> (8 * b)) : 0;
            tr.update(le, 8);
            tr.update(blob + vi.ad_off, vi.ad_len);
        };
        // B. input point; delinearisation scalar z (primitives.py:128-144); operand of z*I
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            TeCoopState& s = cs[item];
            if (s.live && lane == 0) {
                TEExt sum = te_add(TEExt::from_affine(maps[2 * item]), TEExt::from_affine(maps[2 * item + 1]));
                const TEAffine input = te_to_affine(te_dbl(te_dbl(sum)));
                maps[2 * item] = input;
                VrfHash tr;
                transcript(p, input, tr);
                tr.update_byte(0x30);
                uint8_t zb[16];
                vrf_squeeze(tr, zb, 16);
                load_le_limbs8(s.k, zb, 16);
                coop_set_point(s.tab[0], TEExt::from_affine(input));
            }
        }
        DR_BLOCK_SYNC();
        te_straus_coop(ctx, cs, 4, 0);
        // C. I' = G + z*I (first operand of the final Straus); operand of z*O
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            TeCoopState& s = cs[item];
            if (s.live && lane == 0) {
                const TEExt merged_in = te_add(TEExt::from_affine(su.generator), coop_get_point(s.acc));
                coop_set_point(s.tab2[0], merged_in);  // parked: the next multiplication only uses tab
                coop_set_point(s.tab[0], TEExt::from_affine(pts[(size_t)npts * p]));
            }
        }
        DR_BLOCK_SYNC();
        te_straus_coop(ctx, cs, 4, 0);
        // D. O' = PK + z*O; operands of s*I' - c*O'
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            TeCoopState& s = cs[item];
            if (s.live && lane == 0) {
                const uint8_t* pr = proofs + (size_t)plen * p;
                const TEExt merged_out = te_add(TEExt::from_affine(pts[(size_t)npts * p + npts - 1]), coop_get_point(s.acc));
                const TEExt merged_in = coop_get_point(s.tab2[0]);
                coop_set_point(s.tab[0], merged_in);
                coop_set_point(s.tab2[0], te_neg(merged_out));
                load_le_limbs8(s.k, pr + (thin ? 64 : 48), 32);  // s
                if (thin) {  // c from the transcript extended by R
                    VrfHash tr;
                    transcript(p, maps[2 * item], tr);
                    tr.update_byte(0x40);
                    sha_absorb_point(tr, pts[(size_t)npts * p + 1]);
                    uint8_t cb[16];
                    vrf_squeeze(tr, cb, 16);
                    load_le_limbs8(s.k2, cb, 16);
                } else {
                    load_le_limbs8(s.k2, pr + 32, 16);  // c
                }
            }
        }
        DR_BLOCK_SYNC();
        te_straus_coop(ctx, cs, 8, 4);
        // E. verdict
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t item = t / COOP_LANES, lane = t % COOP_LANES, p = ctx.bx * items + item;
            TeCoopState& s = cs[item];
            if (s.live && lane == 0) {
                const uint8_t* pr = proofs + (size_t)plen * p;
                const TEExt res = coop_get_point(s.acc);  // s*I' - c*O'
                bool valid;
                if (thin) {
                    valid = te_ext_eq_affine(res, pts[(size_t)npts * p + 1]);
                } else {
                    VrfHash tr;
                    transcript(p, maps[2 * item], tr);
                    tr.update_byte(0x40);
                    sha_absorb_point(tr, te_to_affine(res));
                    uint8_t cb[16];
                    vrf_squeeze(tr, cb, 16);
                    valid = true;
                    for (int b = 0; b < 16; b++) valid = valid && (cb[b] == pr[32 + b]);
                }
                status[p] = valid ? 0u : ST_PEDERSEN_BAD;
            }
        }
    }
};

// ---- standalone provers (pedersen/vrf.py:86-126, ietf/tiny.py:35-70), one thread per item -------------------------
struct PedersenProveStandaloneBody {  // blinding32: optional n x 32 bytes, the blinding factor b of every proof (vrf.py:144-148)
    DR_HD void operator()(const BlockCtx& ctx, SuiteDev su, const VerifyInput* in, const uint8_t* blob, const uint8_t* sks32, uint32_t count, uint8_t* out192,
                          uint8_t* blinding32) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < count) {
                const VerifyInput& vi = in[i];
                TEAffine pk, blinded;
                uint32_t braw[8];
                pedersen_prove_core(su, sks32 + 32 * (size_t)i, blob + vi.in_off, vi.in_len, blob + vi.ad_off, vi.ad_len, out192 + 192 * (size_t)i, pk, blinded, braw);
                if (blinding32)
                    for (int b = 0; b < 32; b++) blinding32[32 * (size_t)i + b] = (uint8_t)(braw[b >> 2] >> (8 * (b & 3)));
            }
        }
    }
};

struct IetfProveBody {  // thin == 0: O | c | s (80 bytes);  thin != 0: O | R | s (96 bytes)
    DR_HD void operator()(const BlockCtx& ctx, SuiteDev su, uint32_t thin, const VerifyInput* in, const uint8_t* blob, const uint8_t* sks32, uint32_t count,
                          uint8_t* out) const {
        const uint32_t plen = thin ? 96 : 80;
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < count) {
                const VerifyInput& vi = in[i];
                Fn x = fp_from_le_bytes_mod<Fn>(sks32 + 32 * (size_t)i, 32);
                uint32_t xr[8];
                fn_raw_limbs(xr, x);
                TEAffine input = vrf_encode_to_curve(su, blob + vi.in_off, vi.in_len);
                TEAffine pk, output;
                te_to_affine2(te_mul_fixed(su.g_tab, xr), te_mul_glv(input, xr), pk, output);
                VrfHash tr;
                tr.init(su.hash_kind);
                tr.update(su.suite_id, su.suite_id_len);
                tr.update_byte(thin ? 0x01 : 0x00);
                uint8_t le[8] = {2, 0, 0, 0, 0, 0, 0, 0};
                tr.update(le, 8);
                sha_absorb_point(tr, su.generator);
                sha_absorb_point(tr, pk);
                sha_absorb_point(tr, input);
                sha_absorb_point(tr, output);
                for (int b = 0; b < 8; b++) le[b] = b < 4 ? (uint8_t)(vi.ad_len >> (8 * b)) : 0;
                tr.update(le, 8);
                tr.update(blob + vi.ad_off, vi.ad_len);
                VrfHash td = tr;
                td.update_byte(0x30);
                uint8_t zb[16];
                vrf_squeeze(td, zb, 16);
                uint32_t z[8];
                load_le_limbs8(z, zb, 16);
                TEAffine min = te_to_affine(te_add(TEExt::from_affine(su.generator), te_mul_raw(input, z, 4)));
                Fn k = vrf_nonce(tr, x);
                TEAffine r = te_mul_fn(min, k);
                tr.update_byte(0x40);
                sha_absorb_point(tr, r);
                uint8_t* o = out + (size_t)plen * i;
                uint8_t cb[16];
                vrf_squeeze(tr, cb, 16);
                Fn c = fp_from_le_bytes_mod<Fn>(cb, 16);
                te_encode(o, output);
                if (thin) {
                    te_encode(o + 32, r);
                    fn_to_le_bytes(o + 64, k + c * x);
                } else {
                    for (int b = 0; b < 16; b++) o[32 + b] = cb[b];
                    fn_to_le_bytes(o + 48, k + c * x);
                }
            }
        }
    }
};

// ---- ring-proof verifier ------------------------------------------------------------------------------------
struct VerifierKeyDev {
    uint32_t N, logN;
    Fr omega, w_last, n_inv;
    Fr tail[4];         // coefficients of (X - w^(N-1))(X - w^(N-2))(X - w^(N-3))
    TEAffine seed;      // accumulator base
    G1Affine fixed[4];  // C_px, C_py, C_s, [1]_1
    G2Affine g2[2];     // [1]_2, [tau]_2
    PairingConsts pc;
    const LineCoeffs* lines;  // [2][MILLER_LINES] precomputed Miller-loop lines of g2[0], g2[1] (device memory)
    Shake128 prefix;    // transcript after absorbing the verifier key (root.py:54-71)
};

constexpr int VERIFY_TERMS = 13;  // scalar multiplications per proof (see RingVerifyAlgebraBody)

struct VerifyState {
    uint32_t status;
    G1Affine g1[7];      // C_b, C_accip, C_accx, C_accy, C_q, Phi_zeta, Phi_zeta_omega
    uint8_t outside[7];  // g1[j] decoded but not in G1 (g1_in_subgroup): its terms take a full-scalar multiplication
    Fr sc[VERIFY_TERMS];
    G1 term[2 * VERIFY_TERMS];  // sc[j] * base_j as two GLV halves: term[2j] = k1 * P, term[2j + 1] = k2 * phi(P)
};

// 7 G1 decompressions per payload, one thread per point (proof_payload.py:93-118, kzg.py:137-144)
struct PayloadG1DecodeBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* payloads, uint32_t stride, uint32_t count, VerifyState* vs) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < 7 * count) {
                uint32_t p = i / 7, j = i % 7;
                const uint32_t off[7] = {0, 48, 96, 144, 416, 496, 544};
                G1Affine a;
                bool good = g1_decode(a, payloads + (size_t)stride * p + off[j], 48);
                vs[p].g1[j] = good ? a : G1Affine::inf();
                if (!good) vs[p].status = ST_MALFORMED;  // racing writers store the same value
            }
        }
    }
};

// G1 membership of the decoded points, one thread per point: outside[j] sends g1[j]'s terms to a full-scalar multiplication
// (RingVerifyTermsBody).  Nothing else reads it, so it runs on a side stream next to RingVerifyAlgebraBody.
struct PayloadG1SubgroupBody {
    DR_HD void operator()(const BlockCtx& ctx, uint32_t count, VerifyState* vs) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < 7 * count) {
                uint32_t p = i / 7, j = i % 7;
                vs[p].outside[j] = g1_in_subgroup(vs[p].g1[j]) ? 0 : 1;  // infinity (and a malformed point, stored as infinity) is in G1
            }
        }
    }
};

// Challenges + scalar algebra for one payload (phases.py:46-69, verify.py:51-210), then the 13 scalars of the
// random-linear-combined check with coefficients (ra, rb) for the proof's two openings:
//   lhs = sum_j sc[j]*g1[j] (j<7) + sc[9]*C_px + sc[10]*C_py + sc[11]*C_s + sc[12]*[1]_1,  rhs = sc[7]*Phi_zeta + sc[8]*Phi_zeta_omega
//   accept  <=>  e(lhs, [1]_2) == e(rhs, [tau]_2)
struct RingVerifyAlgebraBody {
    DR_HD void operator()(const BlockCtx& ctx, VerifierKeyDev vk, const uint8_t* payloads, uint32_t stride, const TEAffine* relations, uint32_t rel_stride,
                          const uint8_t* coeffs_le32, uint32_t count, VerifyState* vs) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t p = ctx.bx * ctx.nthreads + t;
            if (p < count) {
                VerifyState& s = vs[p];
                const uint8_t* pl = payloads + (size_t)stride * p;
                // evaluations px, py, s, b, accip, accx, accy at zeta and L(zeta w): canonical scalars only
                Fr ev[8];
                bool canon = true;
                for (int i = 0; i < 8; i++) {
                    Fr raw;
                    fr_from_le_bytes_raw(raw, pl + (i < 7 ? 192 + 32 * i : 464));
                    canon = canon && raw.is_canonical_raw();
                    ev[i] = raw.to_mont();
                }
                if (!canon) s.status |= ST_MALFORMED;
                Fr ra, rb;
                fr_from_le_bytes_raw(ra, coeffs_le32 + 64 * (size_t)p);
                fr_from_le_bytes_raw(rb, coeffs_le32 + 64 * (size_t)p + 32);
                ra = ra.to_mont();
                rb = rb.to_mont();
                const TEAffine rel = relations[(size_t)rel_stride * p];
                // ---- transcript
                Shake128 tr = vk.prefix;
                shake_absorb_label(tr, "instance", 8);
                shake_absorb_fr(tr, rel.x);
                shake_absorb_fr(tr, rel.y);
                tr.absorb_be32(64);
                shake_absorb_label(tr, "committed_cols", 14);
                for (int i = 0; i < 4; i++) shake_absorb_g1(tr, s.g1[i]);
                tr.absorb_be32(4 * 96);
                Fr alpha[7], zeta, nu[8];
                shake_challenges(tr, "constraints_aggregation", 23, alpha, 7);
                shake_absorb_label(tr, "quotient", 8);
                shake_absorb_g1(tr, s.g1[4]);
                tr.absorb_be32(96);
                shake_challenges(tr, "evaluation_point", 16, &zeta, 1);
                shake_absorb_label(tr, "register_evaluations", 20);
                tr.absorb(pl + 192, 7 * 32);
                tr.absorb_be32(7 * 32);
                shake_absorb_label(tr, "shifted_linearization_evaluation", 32);
                tr.absorb(pl + 464, 32);
                tr.absorb_be32(32);
                shake_challenges(tr, "kzg_aggregation", 15, nu, 8);
                // ---- verify.py:51-144
                const Fr one = Fr::one();
                Fr zn = zeta;
                for (uint32_t i = 0; i < vk.logN; i++) zn = zn.sqr();
                Fr zn1 = zn - one, zm1 = zeta - one, zml = zeta - vk.w_last;
                // three inversions by Montgomery's trick; a zero denominator makes the reference raise -> invalid
                bool degenerate = zn1.is_zero();
                Fr d1 = zm1.is_zero() ? one : zm1, d2 = zml.is_zero() ? one : zml, d0 = degenerate ? one : zn1;
                Fr p01 = d0 * d1;
                Fr inv_all = (p01 * d2).inv();
                Fr inv_zml = inv_all * p01;
                Fr inv01 = inv_all * d2;
                Fr inv_zn1 = inv01 * d1, inv_zm1 = inv01 * d0;
                Fr l0 = zm1.is_zero() ? one : vk.n_inv * zn1 * inv_zm1;
                Fr ln = zml.is_zero() ? one : vk.w_last * vk.n_inv * zn1 * inv_zml;
                const Fr &x2 = ev[0], &y2 = ev[1], &sz = ev[2], &b = ev[3], &aip = ev[4], &x1 = ev[5], &y1 = ev[6], &lzw = ev[7];
                Fr omb = one - b;
                Fr x1y1 = x1 * y1, x2y2 = x2 * y2;
                TEAffine rps = te_to_affine(te_add(TEExt::from_affine(vk.seed), TEExt::from_affine(rel)));
                Fr cv[7];
                cv[0] = (aip + b * sz).neg() * zml;
                cv[1] = (b * (x1y1 + x2y2).neg() + omb * x1.neg()) * zml;
                cv[2] = (b * (x1y1 - x2y2).neg() + omb * y1.neg()) * zml;
                cv[3] = b * omb;
                cv[4] = (x1 - vk.seed.x) * l0 + (x1 - rps.x) * ln;
                cv[5] = (y1 - vk.seed.y) * l0 + (y1 - rps.y) * ln;
                cv[6] = aip * l0 + (aip - one) * ln;
                Fr lin = Fr::zero();
                for (int i = 0; i < 7; i++) lin = lin + alpha[i] * cv[i];
                Fr prod = ((zeta + vk.tail[2]) * zeta + vk.tail[1]) * zeta + vk.tail[0];
                Fr q_zeta = (lin + lzw) * prod * inv_zn1;
                Fr agg = nu[0] * x2 + nu[1] * y2 + nu[2] * sz + nu[3] * b + nu[4] * aip + nu[5] * x1 + nu[6] * y1 + nu[7] * q_zeta;
                Fr cx = b * (y1 * y2 - fr_mul5(x1 * x2)) + omb;
                Fr cy = b * (x1 * y2 - x2 * y1) + omb;
                Fr s_ip = alpha[0] * zml, s_x = alpha[1] * (cx * zml), s_y = alpha[2] * (cy * zml);
                Fr zeta_omega = zeta * vk.omega;
                if (degenerate) s.status |= ST_PEDERSEN_BAD;
                // ---- kzg.py:56-81 with this proof's two coefficients
                s.sc[0] = ra * nu[3];
                s.sc[1] = ra * nu[4] + rb * s_ip;
                s.sc[2] = ra * nu[5] + rb * s_x;
                s.sc[3] = ra * nu[6] + rb * s_y;
                s.sc[4] = ra * nu[7];
                s.sc[5] = ra * zeta;
                s.sc[6] = rb * zeta_omega;
                s.sc[7] = ra;
                s.sc[8] = rb;
                s.sc[9] = ra * nu[0];
                s.sc[10] = ra * nu[1];
                s.sc[11] = ra * nu[2];
                s.sc[12] = (ra * agg + rb * lzw).neg();
            }
        }
    }
};

// k * P for a Montgomery Fr scalar and an affine base: 4-bit windows over the affine multiples 1P .. 15P (one shared
// inversion), so every window costs 4 doublings + 1 mixed addition
DR_HD_COLD G1 g1_mul_raw(const G1Affine& p, const uint32_t* k, int nlimbs);
DR_HD_COLD G1 g1_mul_fr(const G1Affine& p, const Fr& k_mont) {
    Fr k = k_mont.from_mont();
    return g1_mul_raw(p, k.v, 8);
}
// k: raw little-endian limbs
DR_HD_COLD G1 g1_mul_raw(const G1Affine& p, const uint32_t* k, int nlimbs) {
    if (p.is_inf()) return G1::inf();
    G1 proj[16];
    proj[1] = G1::from_affine(p);
#pragma unroll 1
    for (int i = 2; i < 16; i++) {
        if (i & 1) {
            proj[i] = proj[i - 1];
            g1_madd(proj[i], p);
        } else {
            proj[i] = g1_dbl(proj[i >> 1]);
        }
    }
    // batch-normalise 2P .. 15P
    G1Affine tab[16];
    Fq pre[16], den[16];
    Fq acc = Fq::one();
#pragma unroll 1
    for (int i = 2; i < 16; i++) {
        pre[i] = acc;
        den[i] = proj[i].ZZ * proj[i].ZZZ;
        acc = acc * den[i];
    }
    Fq inv = acc.inv();
    tab[1] = p;
#pragma unroll 1
    for (int i = 15; i >= 2; i--) {
        Fq di = inv * pre[i];
        inv = inv * den[i];
        tab[i] = {proj[i].X * (di * proj[i].ZZZ), proj[i].Y * (di * proj[i].ZZ)};
    }
    G1 r = G1::inf();
#pragma unroll 1
    for (int i = nlimbs - 1; i >= 0; i--) {
#pragma unroll 1
        for (int sft = 28; sft >= 0; sft -= 4) {
            if (!r.is_inf()) r = g1_dbl(g1_dbl(g1_dbl(g1_dbl(r))));
            uint32_t d = (k[i] >> sft) & 15;
            if (d) g1_madd(r, tab[d]);
        }
    }
    return r;
}

// one thread per (proof, term, GLV half): sc * P = k1 * P + k2 * phi(P) with 128-bit k1, k2 (msm.cuh glv_half), phi(x, y) = (beta x, y):
// half the doublings of a 255-bit multiplication, on twice the threads.  A decoded point outside G1 takes sc * P whole on the first
// half's thread (the split is exact only on G1; g1_mul_raw's affine table assumes no multiple 2P .. 15P is infinity, which a
// small-order component breaks); the fixed points are commitments over the SRS, in G1.
struct RingVerifyTermsBody {
    DR_HD void operator()(const BlockCtx& ctx, VerifierKeyDev vk, uint32_t count, VerifyState* vs) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < 2 * VERIFY_TERMS * count) {
                uint32_t p = i / (2 * VERIFY_TERMS), r = i % (2 * VERIFY_TERMS), j = r >> 1, h = r & 1;
                VerifyState& s = vs[p];
                const uint32_t src = j < 7 ? j : j - 2;  // index into s.g1 for j < 9
                G1Affine base = j < 9 ? s.g1[src] : vk.fixed[j - 9];
                G1 out = G1::inf();
                if (!(s.status & ST_MALFORMED) && !base.is_inf()) {
                    Fr k = s.sc[j].from_mont();
                    if (j < 9 && s.outside[src]) {
                        if (!h) out = g1_mul_limbs(G1::from_affine(base), k.v);  // XYZZ table: multiples of a small-order point may be infinity
                    } else {
                        uint32_t half[8];
                        glv_half(k.v, h, half);
                        if (h) base.x = base.x * glv_beta();
                        out = g1_mul_raw(base, half, 4);
                    }
                }
                s.term[r] = out;
            }
        }
    }
};

DR_HD void ring_verify_sides(const VerifyState& s, G1& lhs, G1& rhs) {
    lhs = s.term[0];
    for (int j = 1; j < 2 * 7; j++) g1_add(lhs, s.term[j]);
    for (int j = 2 * 9; j < 2 * VERIFY_TERMS; j++) g1_add(lhs, s.term[j]);
    rhs = s.term[2 * 7];
    for (int j = 2 * 7 + 1; j < 2 * 9; j++) g1_add(rhs, s.term[j]);
}

// per-item verdicts: one 32-thread block per proof runs the warp-cooperative pairing check.
// extra_status: Pedersen status per proof (or null).
DR_HD size_t ring_verify_warp_smem() { return sizeof(PairingWarpState) + 2 * sizeof(G1) + 16; }
struct RingVerifyFinishBody {
    DR_HD void operator()(const BlockCtx& ctx, VerifierKeyDev vk, uint32_t count, const VerifyState* vs, const uint32_t* extra_status, uint8_t* verdict) const {
        PairingWarpState* st = (PairingWarpState*)ctx.smem;
        G1* P = (G1*)(ctx.smem + ((sizeof(PairingWarpState) + 15) / 16) * 16);
        const uint32_t p = ctx.bx;
        if (p >= count) return;
        const VerifyState& s = vs[p];
        const uint32_t stt = s.status | (extra_status ? extra_status[p] : 0u);
        if (stt) {  // uniform over the block
            DR_THREAD_LOOP(t, ctx) {
                if (t == 0) verdict[p] = (stt & ST_MALFORMED) ? 2 : 0;
            }
            return;
        }
        DR_THREAD_LOOP(t, ctx) {
            if (t < 2) {  // both lanes fold one side (same code path: no divergence)
                const int lo = t == 0 ? 0 : 2 * 7, mid = t == 0 ? 2 * 7 : 2 * 9, lo2 = t == 0 ? 2 * 9 : 0, hi2 = t == 0 ? 2 * VERIFY_TERMS : 0;
                G1 acc = s.term[lo];
                for (int j = lo + 1; j < mid; j++) g1_add(acc, s.term[j]);
                for (int j = lo2; j < hi2; j++) g1_add(acc, s.term[j]);
                P[t] = t == 0 ? acc : g1_neg(acc);  // e(lhs, [1]_2) * e(-rhs, [tau]_2) == 1
            }
        }
        DR_BLOCK_SYNC();
        pairing_product_is_one_warp(ctx, st, P, vk.lines, vk.pc);
        DR_THREAD_LOOP(t, ctx) {
            if (t == 0) verdict[p] = st->verdict ? 1 : 0;
        }
    }
};

// aggregated check (RingVRF.batch_verify, vrf/ring/vrf.py:239-283), stage 1: every block folds a strided share of the proofs'
// two sides into one (lhs, rhs) pair; verdict[p] carries the per-item decode / Pedersen status (1 ok, 0 invalid, 2 malformed).
struct RingVerifyPartialSumBody {
    DR_HD void operator()(const BlockCtx& ctx, uint32_t count, const VerifyState* vs, const uint32_t* extra_status, uint8_t* verdict, G1* partial,
                          uint32_t* any_bad) const {
        G1* sm = (G1*)ctx.smem;  // 2 * nthreads
        const uint32_t stride_all = ctx.gx * ctx.nthreads;
        DR_THREAD_LOOP(t, ctx) {
            G1 lhs = G1::inf(), rhs = G1::inf();
#pragma unroll 1
            for (uint32_t p = ctx.bx * ctx.nthreads + t; p < count; p += stride_all) {
                const VerifyState& s = vs[p];
                uint32_t st = s.status | (extra_status ? extra_status[p] : 0u);
                verdict[p] = (st & ST_MALFORMED) ? 2 : st ? 0 : 1;
                if (st) {
                    *any_bad = 1;  // racing writers store the same value
                } else {
                    G1 l, r;
                    ring_verify_sides(s, l, r);
                    g1_add(lhs, l);
                    g1_add(rhs, r);
                }
            }
            sm[t] = lhs;
            sm[ctx.nthreads + t] = rhs;
        }
        DR_BLOCK_SYNC();
        for (uint32_t stride = ctx.nthreads >> 1; stride > 0; stride >>= 1) {
            DR_STRIDE_LOOP(t, stride, ctx) {
                G1 a = sm[t];
                g1_add(a, sm[t + stride]);
                sm[t] = a;
                G1 b = sm[ctx.nthreads + t];
                g1_add(b, sm[ctx.nthreads + t + stride]);
                sm[ctx.nthreads + t] = b;
            }
            DR_BLOCK_SYNC();
        }
        DR_THREAD_LOOP(t, ctx) {
            if (t == 0) {
                partial[2 * ctx.bx] = sm[0];
                partial[2 * ctx.bx + 1] = sm[ctx.nthreads];
            }
        }
    }
};
// Large aggregated batches: instead of 13 scalar multiplications per proof (RingVerifyTermsBody), the two sides become two
// variable-base MSMs (pippenger.cuh): lhs over 7 points per proof + the 4 fixed points, rhs over 2 points per proof.
// This kernel lays out the operands: points, canonical little-endian scalars, and per-block sums of the fixed scalars.
struct RingVerifyGatherBody {
    DR_HD void operator()(const BlockCtx& ctx, uint32_t count, const VerifyState* vs, const uint32_t* extra_status, uint8_t* verdict, G1Affine* lhs_pts, uint8_t* lhs_sc,
                          G1Affine* rhs_pts, uint8_t* rhs_sc, Fr* fixed_partial, uint32_t* any_bad) const {
        Fr* sm = (Fr*)ctx.smem;  // 4 * nthreads
        DR_THREAD_LOOP(t, ctx) {
            uint32_t p = ctx.bx * ctx.nthreads + t;
            Fr f[4] = {Fr::zero(), Fr::zero(), Fr::zero(), Fr::zero()};
            if (p < count) {
                const VerifyState& s = vs[p];
                uint32_t st = s.status | (extra_status ? extra_status[p] : 0u);
                verdict[p] = (st & ST_MALFORMED) ? 2 : st ? 0 : 1;
                if (st) *any_bad = 1;  // racing writers store the same value
                for (int j = 0; j < 7; j++) {
                    lhs_pts[7 * (size_t)p + j] = st ? G1Affine::inf() : s.g1[j];
                    fr_to_le_bytes_raw(lhs_sc + 32 * (7 * (size_t)p + j), st ? Fr::zero() : s.sc[j].from_mont());
                }
                for (int j = 0; j < 2; j++) {
                    rhs_pts[2 * (size_t)p + j] = st ? G1Affine::inf() : s.g1[5 + j];
                    fr_to_le_bytes_raw(rhs_sc + 32 * (2 * (size_t)p + j), st ? Fr::zero() : s.sc[7 + j].from_mont());
                }
                if (!st)
                    for (int j = 0; j < 4; j++) f[j] = s.sc[9 + j];
            }
            for (int j = 0; j < 4; j++) sm[j * ctx.nthreads + t] = f[j];
        }
        DR_BLOCK_SYNC();
        for (uint32_t stride = ctx.nthreads >> 1; stride > 0; stride >>= 1) {
            DR_STRIDE_LOOP(t, stride, ctx) {
                for (int j = 0; j < 4; j++) sm[j * ctx.nthreads + t] = sm[j * ctx.nthreads + t] + sm[j * ctx.nthreads + t + stride];
            }
            DR_BLOCK_SYNC();
        }
        DR_THREAD_LOOP(t, ctx) {
            if (t < 4) fixed_partial[4 * (size_t)ctx.bx + t] = sm[t * ctx.nthreads];
        }
    }
};
// appends the 4 fixed points with their summed scalars after the 7 * count per-proof entries
struct RingVerifyFixedBody {
    DR_HD void operator()(const BlockCtx& ctx, VerifierKeyDev vk, uint32_t count, const Fr* fixed_partial, uint32_t nparts, G1Affine* lhs_pts, uint8_t* lhs_sc) const {
        DR_THREAD_LOOP(t, ctx) {
            if (t < 4) {
                Fr acc = Fr::zero();
                for (uint32_t i = 0; i < nparts; i++) acc = acc + fixed_partial[4 * (size_t)i + t];
                lhs_pts[7 * (size_t)count + t] = vk.fixed[t];
                fr_to_le_bytes_raw(lhs_sc + 32 * (7 * (size_t)count + t), acc.from_mont());
            }
        }
    }
};
// the two MSM results as the (lhs, rhs) pair RingVerifyAggregateBody folds
struct RingVerifySidesFromAffineBody {
    DR_HD void operator()(const BlockCtx& ctx, const G1Affine* sides, G1* partial) const {
        DR_THREAD_LOOP(t, ctx) {
            if (t < 2) partial[t] = G1::from_affine(sides[t]);
        }
    }
};

// stage 2: one block folds the partial pairs and runs the single pairing check
struct RingVerifyAggregateBody {
    DR_HD void operator()(const BlockCtx& ctx, VerifierKeyDev vk, const G1* partial, uint32_t nparts, const uint32_t* any_bad, uint32_t* all_ok) const {
        PairingWarpState* st = (PairingWarpState*)ctx.smem;
        G1* P = (G1*)(ctx.smem + ((sizeof(PairingWarpState) + 15) / 16) * 16);
        DR_THREAD_LOOP(t, ctx) {
            if (t < 2) {
                G1 acc = G1::inf();
#pragma unroll 1
                for (uint32_t i = 0; i < nparts; i++) g1_add(acc, partial[2 * i + t]);
                P[t] = t == 0 ? acc : g1_neg(acc);
            }
        }
        DR_BLOCK_SYNC();
        pairing_product_is_one_warp(ctx, st, P, vk.lines, vk.pc);
        DR_THREAD_LOOP(t, ctx) {
            if (t == 0) *all_ok = (!*any_bad && st->verdict) ? 1u : 0u;
        }
    }
};

}  // namespace dr
