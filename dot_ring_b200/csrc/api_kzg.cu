// C ABI, part 6: the rest of the PCS seam (dot_ring/ring_proof/pcs/protocol.py:33-40) -- KZG.open and the pairing side of
// KZG.verify / batch_verify / batch_verify_linear_preconverted (pcs/kzg.py:178-338) against the SRS of the context.
#include "api_internal.cuh"

namespace dr {

// one block per polynomial: y = f(x), then f <- (f - y) / (X - x) in place (pcs/utils.py:27-35).  The value is taken before
// the division overwrites the coefficients.
struct KzgOpenBody {
    DR_HD void operator()(const BlockCtx& ctx, Fr* polys, uint32_t n, const Fr* xs, Fr* ys) const {
        Fr* poly = polys + (size_t)ctx.bx * n;
        const Fr x = xs[ctx.bx];
        Fr y = block_poly_eval(ctx, poly, n, x, (Fr*)ctx.smem);
        DR_THREAD_LOOP(t, ctx) {
            if (t == 0) ys[ctx.bx] = y;
        }
        block_synthetic_div(ctx, poly, n, x, (Fr*)ctx.smem);
    }
};

// one thread per term: out[i] = (scalar_i mod r) * P_i; bad = 1 on a malformed point encoding
struct G1TermMulBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* pts_be96, const Fr* scalars, uint32_t n, G1* out, uint32_t* bad) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < n) {
                G1Affine a;
                if (!g1_decode(a, pts_be96 + 96 * (size_t)i, 96)) {
                    *bad = 1;
                    a = G1Affine::inf();
                }
                out[i] = g1_mul_fr(a, scalars[i]);
            }
        }
    }
};

// fold `n` terms into one XYZZ point: grid (parts); out[part] = sum of a strided share
struct G1FoldBody {
    DR_HD void operator()(const BlockCtx& ctx, const G1* terms, uint32_t n, G1* out, uint32_t out_stride) const {
        G1* sm = (G1*)ctx.smem;
        DR_THREAD_LOOP(t, ctx) {
            G1 acc = G1::inf();
#pragma unroll 1
            for (uint32_t i = ctx.bx * ctx.nthreads + t; i < n; i += ctx.gx * ctx.nthreads) g1_add(acc, terms[i]);
            sm[t] = acc;
        }
        DR_BLOCK_SYNC();
        for (uint32_t stride = ctx.nthreads >> 1; stride > 0; stride >>= 1) {
            DR_STRIDE_LOOP(t, stride, ctx) {
                G1 a = sm[t];
                g1_add(a, sm[t + stride]);
                sm[t] = a;
            }
            DR_BLOCK_SYNC();
        }
        DR_THREAD_LOOP(t, ctx) {
            if (t == 0) out[(size_t)ctx.bx * out_stride] = sm[0];
        }
    }
};

struct G1FromAffineBody {
    DR_HD void operator()(const BlockCtx& ctx, const G1Affine* in, G1* out) const {
        DR_THREAD_LOOP(t, ctx) {
            if (t == 0) *out = G1::from_affine(*in);
        }
    }
};

const LineCoeffs* Srs::pairing_lines() {
    if (!lines.p) {
        G2Affine g2[2];
        for (int i = 0; i < 2; i++)
            if (!g2_decode_uncompressed(g2[i], g2_be192 + 192 * i)) throw Error(DR_EINVAL, "invalid BLS12-381 G2 encoding in SRS");
        std::vector<LineCoeffs> host(2 * MILLER_LINES);
        miller_precompute_lines(g2[0], host.data());
        miller_precompute_lines(g2[1], host.data() + MILLER_LINES);
        lines.alloc(host.size());
        h2d(ctx->stream, lines.p, host.data(), host.size() * sizeof(LineCoeffs));
        stream_sync(ctx->stream);
    }
    return lines.p;
}

// sum_i scalars[i] * points[i] spread over out_pairs[slot + 2p], p < parts (XYZZ): per-term multiplications for short sides, the
// bucket method beyond (its latency floor is a few ms)
static void side_sum(Ctx* ctx, const uint8_t* pts_be96, const uint8_t* scalars_le32, size_t n, G1* out_pairs, uint32_t slot, uint32_t parts, uint32_t* dbad) {
    const uint32_t m = (uint32_t)n;
    DevBuf<uint8_t> dpts(n * 96), dsc(n * 32);
    h2d(ctx->stream, dpts.p, pts_be96, n * 96);
    h2d(ctx->stream, dsc.p, scalars_le32, n * 32);
    if (n >= 4096) {
        DevBuf<G1Affine> aff(n), res(1);
        DevBuf<uint8_t> ok(n);
        launch(ctx->stream, Dim3((m + 63) / 64), 64, 0, G1DecodeBody(), (const uint8_t*)dpts.p, 96u, m, aff.p, ok.p);
        std::vector<uint8_t> okh(n);
        d2h(ctx->stream, okh.data(), ok.p, n);
        stream_sync(ctx->stream);
        for (size_t i = 0; i < n; i++)
            if (!okh[i]) throw Error(DR_EINVAL, "invalid BLS12-381 G1 encoding");
        // scalars may be unreduced: canonicalise on the device
        DevBuf<Fr> fr(n);
        launch(ctx->stream, Dim3((m + 255) / 256), 256, 0, FrToMontBody(), (const uint8_t*)dsc.p, fr.p, n, (uint32_t*)nullptr);
        launch(ctx->stream, Dim3((m + 255) / 256), 256, 0, FrFromMontBody(), (const Fr*)fr.p, dsc.p, n);
        msm_points_device(ctx, aff.p, dsc.p, n, res.p);
        launch(ctx->stream, Dim3(1), 32, 0, G1FromAffineBody(), (const G1Affine*)res.p, out_pairs + slot);  // the other parts stay at infinity
        stream_sync(ctx->stream);
        return;
    }
    DevBuf<Fr> fr(n);
    DevBuf<G1> terms(n);
    launch(ctx->stream, Dim3((m + 255) / 256), 256, 0, FrToMontBody(), (const uint8_t*)dsc.p, fr.p, n, (uint32_t*)nullptr);
    launch(ctx->stream, Dim3((m + 31) / 32), 32, 0, G1TermMulBody(), (const uint8_t*)dpts.p, (const Fr*)fr.p, m, terms.p, dbad);
    launch(ctx->stream, Dim3(parts), 64, 64 * sizeof(G1), G1FoldBody(), (const G1*)terms.p, m, out_pairs + slot, 2u);
    stream_sync(ctx->stream);  // scratch goes out of scope
}

}  // namespace dr

using namespace dr;

extern "C" {

int dr_kzg_open(dr_ctx* c, dr_srs* s, const uint8_t* coeffs_le32, size_t n, size_t batch, const uint8_t* points_le32, uint8_t* proofs_be96, uint8_t* values_le32) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    Srs* srs = (Srs*)s;
    if (!ctx || !srs || (batch && (!points_le32 || !proofs_be96 || !values_le32)) || (n * batch && !coeffs_le32)) throw Error(DR_EINVAL, "bad argument");
    if (n == 0) throw Error(DR_EINVAL, "cannot open the empty polynomial");  // the reference indexes poly[-1] (pcs/utils.py:31)
    if (n > (size_t)srs->n + 1) throw Error(DR_EINVAL, "polynomial degree exceeds SRS size");
    ctx->activate();
    if (!batch) return DR_OK;
    const size_t total = n * batch;
    DevBuf<uint8_t> raw(total * 32), xraw(batch * 32), yraw(batch * 32), enc(batch * 96);
    DevBuf<Fr> poly(total), xs(batch), ys(batch);
    DevBuf<G1Affine> res(batch);
    h2d(ctx->stream, raw.p, coeffs_le32, total * 32);
    h2d(ctx->stream, xraw.p, points_le32, batch * 32);
    launch(ctx->stream, Dim3((uint32_t)((total + 255) / 256)), 256, 0, FrToMontBody(), (const uint8_t*)raw.p, poly.p, total, (uint32_t*)nullptr);
    launch(ctx->stream, Dim3((uint32_t)((batch + 255) / 256)), 256, 0, FrToMontBody(), (const uint8_t*)xraw.p, xs.p, batch, (uint32_t*)nullptr);
    launch(ctx->stream, Dim3((uint32_t)batch), 256, synthetic_div_smem(256), KzgOpenBody(), poly.p, (uint32_t)n, (const Fr*)xs.p, ys.p);
    if (n > 1) {
        commit_device(ctx, srs, poly.p, n, (uint32_t)(n - 1), (uint32_t)batch, res.p);
        launch(ctx->stream, Dim3((uint32_t)((batch + 63) / 64)), 64, 0, G1EncodeBody(), (const G1Affine*)res.p, (uint32_t)batch, enc.p, (uint8_t*)nullptr);
        d2h(ctx->stream, proofs_be96, enc.p, batch * 96);
    } else {
        for (size_t b = 0; b < batch; b++) {  // constant polynomial: empty quotient commits to infinity (kzg.py:167-168)
            memset(proofs_be96 + 96 * b, 0, 96);
            proofs_be96[96 * b] = 0x40;
        }
    }
    launch(ctx->stream, Dim3((uint32_t)((batch + 255) / 256)), 256, 0, FrFromMontBody(), (const Fr*)ys.p, yraw.p, batch);
    d2h(ctx->stream, values_le32, yraw.p, batch * 32);
    stream_sync(ctx->stream);
    DR_API_END
}

int dr_kzg_pairing_check(dr_ctx* c, dr_srs* s, const uint8_t* lhs_points_be96, const uint8_t* lhs_scalars_le32, size_t n_lhs, const uint8_t* rhs_points_be96,
                         const uint8_t* rhs_scalars_le32, size_t n_rhs, int* ok) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    Srs* srs = (Srs*)s;
    if (!ctx || !srs || !ok || (n_lhs && (!lhs_points_be96 || !lhs_scalars_le32)) || (n_rhs && (!rhs_points_be96 || !rhs_scalars_le32))) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    *ok = 0;
    const uint32_t parts = 8;
    DevBuf<G1> pairs(2 * parts);  // (lhs, rhs) interleaved, as RingVerifyAggregateBody folds them
    DevBuf<uint32_t> bad(1), dall(1);
    dev_zero(ctx->stream, bad.p, 4);
    {
        std::vector<G1> inf(2 * parts, G1::inf());
        h2d(ctx->stream, pairs.p, inf.data(), inf.size() * sizeof(G1));
        stream_sync(ctx->stream);
    }
    if (n_lhs) side_sum(ctx, lhs_points_be96, lhs_scalars_le32, n_lhs, pairs.p, 0, parts, bad.p);
    if (n_rhs) side_sum(ctx, rhs_points_be96, rhs_scalars_le32, n_rhs, pairs.p, 1, parts, bad.p);
    uint32_t bad_h = 0, all = 0;
    d2h(ctx->stream, &bad_h, bad.p, 4);
    stream_sync(ctx->stream);
    if (bad_h) throw Error(DR_EINVAL, "invalid BLS12-381 G1 encoding");
    launch(ctx->stream, Dim3(1), 32, ring_verify_warp_smem(), RingVerifyAggregateBody(), srs->pairing_lines(), ctx->pairing_consts(), (const G1*)pairs.p, parts, (const uint32_t*)bad.p, dall.p);
    d2h(ctx->stream, &all, dall.p, 4);
    stream_sync(ctx->stream);
    *ok = (int)all;
    DR_API_END
}

}  // extern "C"
