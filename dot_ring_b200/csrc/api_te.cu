// C ABI, part 4: batched Bandersnatch point operations (decode + subgroup check, scalar multiplication).
#include "api_internal.cuh"
#include "ring.cuh"

namespace dr {

struct TeDecodeBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* in, uint32_t n, int checked, uint8_t* out_xy, uint8_t* ok) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < n) {
                TEAffine p;
                bool good = checked ? te_decode_checked(p, in + 32 * (size_t)i) : te_decode(p, in + 32 * (size_t)i);
                if (!good) p = TEAffine::identity();
                fr_to_le_bytes_raw(out_xy + 64 * (size_t)i, p.x.from_mont());
                fr_to_le_bytes_raw(out_xy + 64 * (size_t)i + 32, p.y.from_mont());
                ok[i] = good ? 1 : 0;
            }
        }
    }
};

// out[i] = (k_i mod n) * P_(i or 0); ok[i] = 0 when the point does not decode
struct TeMulBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* pts, uint32_t n_pts, const uint8_t* ks, uint32_t n, uint8_t* out, uint8_t* ok) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < n) {
                TEAffine p;
                bool good = te_decode(p, pts + 32 * (size_t)(n_pts == 1 ? 0 : i));
                if (good) {
                    Fn k = fp_from_le_bytes_mod<Fn>(ks + 32 * (size_t)i, 32);
                    te_encode(out + 32 * (size_t)i, te_mul_fn(p, k));
                } else {
                    for (int b = 0; b < 32; b++) out[32 * (size_t)i + b] = 0;
                }
                ok[i] = good ? 1 : 0;
            }
        }
    }
};

// sum_i (k_i mod n) * P_i: one scalar multiplication per thread, shared-memory tree per block -> partial[block] (extended coords)
struct TeMsmBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* pts, const uint8_t* ks, uint32_t n, TEExt* partial, uint32_t* bad) const {
        TEExt* sm = (TEExt*)ctx.smem;
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            TEExt acc = TEExt::identity();
            if (i < n) {
                TEAffine p;
                if (te_decode(p, pts + 32 * (size_t)i)) {
                    Fn k = fp_from_le_bytes_mod<Fn>(ks + 32 * (size_t)i, 32);
                    uint32_t kr[8];
                    fn_raw_limbs(kr, k);
                    acc = te_mul_raw(p, kr, 8);
                } else {
                    *bad = 1;  // racing writers store the same value
                }
            }
            sm[t] = acc;
        }
        DR_BLOCK_SYNC();
        for (uint32_t stride = ctx.nthreads >> 1; stride > 0; stride >>= 1) {
            DR_STRIDE_LOOP(t, stride, ctx) { sm[t] = te_add(sm[t], sm[t + stride]); }
            DR_BLOCK_SYNC();
        }
        DR_THREAD_LOOP(t, ctx) {
            if (t == 0) partial[ctx.bx] = sm[0];
        }
    }
};
struct TeMsmFinishBody {  // one block folds the per-block partial sums and encodes the result
    DR_HD void operator()(const BlockCtx& ctx, const TEExt* partial, uint32_t nparts, uint8_t* out32) const {
        TEExt* sm = (TEExt*)ctx.smem;
        DR_THREAD_LOOP(t, ctx) {
            TEExt acc = TEExt::identity();
#pragma unroll 1
            for (uint32_t i = t; i < nparts; i += ctx.nthreads) acc = te_add(acc, partial[i]);
            sm[t] = acc;
        }
        DR_BLOCK_SYNC();
        for (uint32_t stride = ctx.nthreads >> 1; stride > 0; stride >>= 1) {
            DR_STRIDE_LOOP(t, stride, ctx) { sm[t] = te_add(sm[t], sm[t + stride]); }
            DR_BLOCK_SYNC();
        }
        DR_THREAD_LOOP(t, ctx) {
            if (t == 0) te_encode(out32, te_to_affine(sm[0]));
        }
    }
};

}  // namespace dr

using namespace dr;

extern "C" {

// Replaces `dec_point` (dot_ring/vrf/codec.py:39-45) / `CurvePoint.string_to_point` (curve/point.py:178-214)
// for a batch: ok[i] = 0 <=> the reference raises ValueError.  checked != 0 adds the non-identity
// prime-subgroup test of `Curve.valid_point` (curve/curve.py:56-67).
int dr_te_decode_batch(dr_ctx* c, const uint8_t* in32, size_t n, int checked, uint8_t* out_xy64, uint8_t* ok) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || (n && (!in32 || !out_xy64 || !ok))) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (!n) return DR_OK;
    DevBuf<uint8_t> din(n * 32), dout(n * 64), dok(n);
    h2d(ctx->stream, din.p, in32, n * 32);
    launch(ctx->stream, Dim3((uint32_t)((n + 63) / 64)), 64, 0, TeDecodeBody(), (const uint8_t*)din.p, (uint32_t)n, checked, dout.p, dok.p);
    d2h(ctx->stream, out_xy64, dout.p, n * 64);
    d2h(ctx->stream, ok, dok.p, n);
    stream_sync(ctx->stream);
    DR_API_END
}

// Replaces `BandersnatchPoint.__mul__` (dot_ring/curve/specs/bandersnatch.py:177-191) for a batch:
// out[i] = (scalars[i] mod order) * points[i]  (or * points[0] when n_points == 1), 32-byte encodings.
int dr_te_mul_batch(dr_ctx* c, const uint8_t* points32, size_t n_points, const uint8_t* scalars32, size_t n, uint8_t* out32, uint8_t* ok) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || (n && (!points32 || !scalars32 || !out32 || !ok)) || (n_points != 1 && n_points != n)) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (!n) return DR_OK;
    DevBuf<uint8_t> dp(n_points * 32), dk(n * 32), dout(n * 32), dok(n);
    h2d(ctx->stream, dp.p, points32, n_points * 32);
    h2d(ctx->stream, dk.p, scalars32, n * 32);
    launch(ctx->stream, Dim3((uint32_t)((n + 63) / 64)), 64, 0, TeMulBody(), (const uint8_t*)dp.p, (uint32_t)n_points, (const uint8_t*)dk.p, (uint32_t)n, dout.p, dok.p);
    d2h(ctx->stream, out32, dout.p, n * 32);
    d2h(ctx->stream, ok, dok.p, n);
    dev_zero(ctx->stream, dk.p, n * 32);  // the scalars may be secret keys (public-key derivation); the block is recycled
    stream_sync(ctx->stream);
    DR_API_END
}

// Replaces `BandersnatchPoint.msm` (dot_ring/curve/specs/bandersnatch.py:194-286: GLV joint windows for n <= 3,
// `msm_pippenger_signed_native_cy` above; native_field/bandersnatch_te.pyx:257-418): out = sum_i (scalars[i] mod order) * points[i].
// Every point is one thread's windowed multiplication, the partial sums are tree-folded.  DR_EINVAL on an undecodable point.
int dr_te_msm(dr_ctx* c, const uint8_t* points32, const uint8_t* scalars32, size_t n, uint8_t out32[32]) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || !out32 || (n && (!points32 || !scalars32))) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    const uint32_t threads = 64;
    const uint32_t blocks = n ? (uint32_t)((n + threads - 1) / threads) : 1;
    DevBuf<uint8_t> dp(n ? n * 32 : 32), dk(n ? n * 32 : 32), dout(32);
    DevBuf<TEExt> partial(blocks);
    DevBuf<uint32_t> bad(1);
    dev_zero(ctx->stream, bad.p, 4);
    h2d(ctx->stream, dp.p, points32, n * 32);
    h2d(ctx->stream, dk.p, scalars32, n * 32);
    launch(ctx->stream, Dim3(blocks), threads, threads * sizeof(TEExt), TeMsmBody(), (const uint8_t*)dp.p, (const uint8_t*)dk.p, (uint32_t)n, partial.p, bad.p);
    launch(ctx->stream, Dim3(1), threads, threads * sizeof(TEExt), TeMsmFinishBody(), (const TEExt*)partial.p, blocks, dout.p);
    uint32_t bad_h = 0;
    d2h(ctx->stream, &bad_h, bad.p, 4);
    d2h(ctx->stream, out32, dout.p, 32);
    stream_sync(ctx->stream);
    if (bad_h) throw Error(DR_EINVAL, "Invalid point encoding");
    DR_API_END
}
}
