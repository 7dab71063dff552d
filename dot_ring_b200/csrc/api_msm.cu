// C ABI, part 6: variable-base G1 MSM (bucket method) and the 2^11 .. 2^20 sweep over a synthetic SRS.
#include "api_internal.cuh"
#include "pippenger.cuh"

namespace dr {

// window bits minimising W * (n + weight * 2^(c-1)) mixed-addition equivalents.  For large sets a bucket costs
// far more than the 2.8 additions of its arithmetic: the fold / running-sum / window kernels are short dependent chains on few threads
// (measured at 2^20 points: 0.43 ns per bucket addition against ~11 ns per bucket), so the model charges a bucket 16 additions from
// 2^18 points on.  Below, those kernels are latency-bound whatever the bucket count and the plain arithmetic count picks better
// (measured with the endomorphism-split recoding this file used before, profiles/r02_probe_msm_sweep*.json: 3.0 vs 3.4 ms at 2^16,
// 5.1 vs 5.3 ms at 2^18, 11.9 vs 13.3 ms at 2^20).
static uint32_t msm_window_bits(size_t n) {
    uint32_t best = 4;
    double best_cost = 1e300;
    const double weight = n >= ((size_t)1 << 18) ? 16.0 : 2.8;
    for (uint32_t c = 4; c <= 17; c++) {
        double W = (MSM_BITS + c - 1) / c;
        double cost = W * ((double)n + weight * (double)(1u << (c - 1)));
        if (cost < best_cost) {
            best_cost = cost;
            best = c;
        }
    }
    return best;
}

struct MsmWork {
    MsmGeom g{};
    uint32_t segs = 0;
    DevBuf<int32_t> digits;
    DevBuf<uint32_t> count, offset, unit_offset, cursor, totals, refs, block_tot;
    DevBuf<G1> unit_sum, bucket, seg_sum, window_sum;
    DevBuf<G1Affine> result;
    void prepare(size_t n_points) {
        g.n = (uint32_t)n_points;
        const size_t n = n_points;
        g.c = msm_window_bits(n_points);
        g.W = (MSM_BITS + g.c - 1) / g.c;
        g.H = 1u << (g.c - 1);
        segs = (g.H + MSM_SEGMENT - 1) / MSM_SEGMENT;
        const size_t nb = g.buckets();
        digits.ensure((size_t)g.W * n);
        count.ensure(nb);
        offset.ensure(nb);
        unit_offset.ensure(nb);
        cursor.ensure(nb);
        totals.ensure(1);
        refs.ensure((size_t)g.W * n);
        unit_sum.ensure((size_t)g.W * n / MSM_UNIT + nb + 1);  // units <= refs / UNIT + one partial unit per bucket
        bucket.ensure(nb);
        seg_sum.ensure((size_t)g.W * segs);
        window_sum.ensure(g.W);
        block_tot.ensure(2 * ((nb + SCAN_TILE - 1) / SCAN_TILE));
        result.ensure(1);
    }
};

// points: n affine Montgomery points on the device; scalars: n x 32 bytes on the device.  Result in w.result[0].
static void msm_device(Ctx* ctx, MsmWork& w, const G1Affine* points, const uint8_t* scalars_le32) {
    const MsmGeom g = w.g;
    const uint32_t nb = g.buckets();
    Stream st = ctx->stream;
    dev_zero(st, w.count.p, (size_t)nb * 4);
    launch(st, Dim3((g.n + 127) / 128), 128, 0, MsmDigitsBody(), scalars_le32, g, w.digits.p, w.count.p);
    const uint32_t tiles = (nb + SCAN_TILE - 1) / SCAN_TILE;
    launch(st, Dim3(tiles), SCAN_TILE, 4 * SCAN_TILE * sizeof(uint32_t), MsmScanTileBody(), (const uint32_t*)w.count.p, nb, w.offset.p, w.unit_offset.p, w.block_tot.p);
    launch(st, Dim3(1), 32, 0, MsmScanBlocksBody(), w.block_tot.p, tiles, w.totals.p);
    launch(st, Dim3(tiles), SCAN_TILE, 0, MsmScanApplyBody(), nb, (const uint32_t*)w.block_tot.p, w.offset.p, w.unit_offset.p, w.cursor.p);
    launch(st, Dim3((g.n + 127) / 128), 128, 0, MsmScatterBody(), g, (const int32_t*)w.digits.p, (const uint32_t*)w.offset.p, w.cursor.p, w.refs.p);
    // upper bound on the unit count is known on the host; threads beyond totals[0] exit
    const size_t max_units = (size_t)g.W * g.n / MSM_UNIT + nb + 1;
    launch(st, Dim3((uint32_t)((max_units + 63) / 64)), 64, 0, MsmUnitSumBody(), g, points, (const uint32_t*)w.count.p, (const uint32_t*)w.offset.p,
           (const uint32_t*)w.unit_offset.p, (const uint32_t*)w.totals.p, (const uint32_t*)w.refs.p, w.unit_sum.p);
    launch(st, Dim3((nb + 63) / 64), 64, 0, MsmBucketFoldBody(), g, (const uint32_t*)w.count.p, (const uint32_t*)w.unit_offset.p, (const G1*)w.unit_sum.p, w.bucket.p);
    launch(st, Dim3(nb), 64, 64 * sizeof(G1), MsmBucketFoldHeavyBody(), (const uint32_t*)w.count.p, (const uint32_t*)w.unit_offset.p, (const G1*)w.unit_sum.p, w.bucket.p);
    launch(st, Dim3((g.W * w.segs + 63) / 64), 64, 0, MsmSegmentReduceBody(), g, (const G1*)w.bucket.p, w.segs, w.seg_sum.p);
    launch(st, Dim3(g.W), 64, 64 * sizeof(G1), MsmWindowFoldBody(), (const G1*)w.seg_sum.p, w.segs, w.window_sum.p);
    launch(st, Dim3(1), 64, 64 * sizeof(G1), MsmFinalBody(), g, (const G1*)w.window_sum.p, w.result.p);
}

// sum_i scalars[i] * points[i] with every operand already on the device; result (affine) written to *out (device memory)
void msm_points_device(Ctx* ctx, const G1Affine* points, const uint8_t* scalars_le32, size_t n, G1Affine* out) {
    MsmWork w;
    w.prepare(n);
    msm_device(ctx, w, points, scalars_le32);
    d2d(ctx->stream, out, w.result.p, sizeof(G1Affine));
    stream_sync(ctx->stream);  // the work buffers are released on return
}

}  // namespace dr

using namespace dr;

static const uint8_t G1_GENERATOR_BE96[96] = {
    0x17, 0xf1, 0xd3, 0xa7, 0x31, 0x97, 0xd7, 0x94, 0x26, 0x95, 0x63, 0x8c, 0x4f, 0xa9, 0xac, 0x0f, 0xc3, 0x68, 0x8c, 0x4f, 0x97, 0x74, 0xb9, 0x05,
    0xa1, 0x4e, 0x3a, 0x3f, 0x17, 0x1b, 0xac, 0x58, 0x6c, 0x55, 0xe8, 0x3f, 0xf9, 0x7a, 0x1a, 0xef, 0xfb, 0x3a, 0xf0, 0x0a, 0xdb, 0x22, 0xc6, 0xbb,
    0x08, 0xb3, 0xf4, 0x81, 0xe3, 0xaa, 0xa0, 0xf1, 0xa0, 0x9e, 0x30, 0xed, 0x74, 0x1d, 0x8a, 0xe4, 0xfc, 0xf5, 0xe0, 0x95, 0xd5, 0xd0, 0x0a, 0xf6,
    0x00, 0xdb, 0x18, 0xcb, 0x2c, 0x04, 0xb3, 0xed, 0xd0, 0x3c, 0xc7, 0x44, 0xa2, 0x88, 0x8a, 0xe4, 0x0c, 0xaa, 0x23, 0x29, 0x46, 0xc5, 0xe7, 0xe1};

static uint64_t splitmix64_next(uint64_t& x) {
    uint64_t z = (x += 0x9E3779B97F4A7C15ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

extern "C" {

int dr_g1_msm(dr_ctx* c, const uint8_t* points_be96, const uint8_t* scalars_le32, size_t n, uint8_t out_be96[96]) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || !out_be96 || (n && (!points_be96 || !scalars_le32)) || n >= (1u << 30)) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (n == 0) {
        memset(out_be96, 0, 96);
        out_be96[0] = 0x40;
        return DR_OK;
    }
    DevBuf<uint8_t> raw(n * 96), sc(n * 32), ok(n), enc(96);
    DevBuf<G1Affine> pts(n);
    h2d(ctx->stream, raw.p, points_be96, n * 96);
    h2d(ctx->stream, sc.p, scalars_le32, n * 32);
    launch(ctx->stream, Dim3((uint32_t)((n + 63) / 64)), 64, 0, G1DecodeBody(), (const uint8_t*)raw.p, 96u, (uint32_t)n, pts.p, ok.p);
    std::vector<uint8_t> okh(n);
    d2h(ctx->stream, okh.data(), ok.p, n);
    stream_sync(ctx->stream);
    for (size_t i = 0; i < n; i++)
        if (!okh[i]) throw Error(DR_EINVAL, "invalid BLS12-381 G1 encoding");
    MsmWork w;
    w.prepare(n);
    msm_device(ctx, w, pts.p, sc.p);
    launch(ctx->stream, Dim3(1), 32, 0, G1EncodeBody(), (const G1Affine*)w.result.p, 1u, enc.p, (uint8_t*)nullptr);
    d2h(ctx->stream, out_be96, enc.p, 96);
    stream_sync(ctx->stream);
    DR_API_END
}

int dr_g1_synthetic_srs(dr_ctx* c, const uint8_t tau_le32[32], size_t offset, size_t n, uint8_t* out_be96) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || !tau_le32 || (n && !out_be96) || offset + n >= (1u << 30)) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (!n) return DR_OK;
    Fr tau;
    fr_from_le_bytes_raw(tau, tau_le32);
    if (!tau.is_canonical_raw()) throw Error(DR_EINVAL, "tau is not canonical");
    tau = tau.to_mont();
    G1Affine gen;
    if (!g1_decode(gen, G1_GENERATOR_BE96, 96)) throw Error(DR_ESTATE, "generator decode failed");
    DevBuf<G1Affine> pts(n);
    DevBuf<uint8_t> enc(n * 96);
    launch(ctx->stream, Dim3((uint32_t)((n + 63) / 64)), 64, 0, SyntheticSrsBody(), gen, tau, (uint32_t)offset, (uint32_t)n, pts.p);
    launch(ctx->stream, Dim3((uint32_t)((n + 63) / 64)), 64, 0, G1EncodeBody(), (const G1Affine*)pts.p, (uint32_t)n, enc.p, (uint8_t*)nullptr);
    d2h(ctx->stream, out_be96, enc.p, n * 96);
    stream_sync(ctx->stream);
    DR_API_END
}

int dr_g1_msm_bench(dr_ctx* c, size_t n, int iters, uint64_t seed, int distribution, const uint8_t tau_le32[32], float* ms_per_iter, uint32_t* window_bits,
                    uint8_t out_be96[96]) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || n == 0 || n >= (1u << 30) || iters <= 0 || !tau_le32) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    Fr tau;
    fr_from_le_bytes_raw(tau, tau_le32);
    if (!tau.is_canonical_raw()) throw Error(DR_EINVAL, "tau is not canonical");
    tau = tau.to_mont();
    G1Affine gen;
    if (!g1_decode(gen, G1_GENERATOR_BE96, 96)) throw Error(DR_ESTATE, "generator decode failed");
    DevBuf<G1Affine> pts(n);
    launch(ctx->stream, Dim3((uint32_t)((n + 63) / 64)), 64, 0, SyntheticSrsBody(), gen, tau, 0u, (uint32_t)n, pts.p);
    // scalars: 0 uniform below 2^254, 1 all ones, 2 bits {0, 1} (witness-like worst case for bucket skew)
    std::vector<uint8_t> host(n * 32, 0);
    uint64_t st = seed;
    for (size_t i = 0; i < n; i++) {
        if (distribution == 0) {
            uint64_t wv[4] = {splitmix64_next(st), splitmix64_next(st), splitmix64_next(st), splitmix64_next(st) >> 2};
            memcpy(&host[32 * i], wv, 32);
        } else if (distribution == 1) {
            host[32 * i] = 1;
        } else {
            host[32 * i] = (uint8_t)(splitmix64_next(st) & 1);
        }
    }
    DevBuf<uint8_t> sc(n * 32), enc(96);
    h2d(ctx->stream, sc.p, host.data(), n * 32);
    MsmWork w;
    w.prepare(n);
    if (window_bits) *window_bits = w.g.c;
    msm_device(ctx, w, pts.p, sc.p);  // warm-up
    stream_sync(ctx->stream);
    float ms = 0;
    dr_ctx_timer_start(c);
    for (int it = 0; it < iters; it++) msm_device(ctx, w, pts.p, sc.p);
    dr_ctx_timer_stop(c, &ms);
    if (ms_per_iter) *ms_per_iter = ms / iters;
    if (out_be96) {
        launch(ctx->stream, Dim3(1), 32, 0, G1EncodeBody(), (const G1Affine*)w.result.p, 1u, enc.p, (uint8_t*)nullptr);
        d2h(ctx->stream, out_be96, enc.p, 96);
        stream_sync(ctx->stream);
    }
    DR_API_END
}

}  // extern "C"
