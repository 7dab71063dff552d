// C ABI, part 2: arithmetic-layer self-test hooks and integer-pipe micro-benchmarks.
//
// dr_field_op runs element-wise field operations on the device so that the PTX carry-chain kernels
// can be compared against Python big integers from the test-suite (the reference's equivalent is
// tests/test_curve_ops/test_native_field.py: 100 random add/sub/mul vs Python ints).
// dr_microbench measures the integer-pipe ceilings that the MSM / scalar-mul rooflines are quoted
// against (SURVEY.md section 8d: "IMAD_peak must be measured on the box").
#include "api_internal.cuh"

namespace dr {

template <class F>
struct FieldOpBody {
    DR_HD void operator()(const BlockCtx& ctx, int op, const F* a, const F* b, F* out, uint32_t count) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < count) {
                F x = a[i].to_mont(), y = b[i].to_mont(), r = F::zero();
                switch (op) {
                    case 0: r = x * y; break;
                    case 1: r = x + y; break;
                    case 2: r = x - y; break;
                    case 3: r = x.inv(); break;
                    case 4: r = x.sqr(); break;
                    case 5: r = x.neg(); break;
                }
                out[i] = r.from_mont();
            }
        }
    }
};

#if !defined(DR_HOST_EMULATION)
// ---- micro-benchmarks (CUDA only) ------------------------------------------------------------------
__global__ void mb_imad32(uint32_t* out, uint32_t seed, int iters) {
    uint32_t a0 = seed + threadIdx.x, a1 = a0 * 3, a2 = a0 * 5, a3 = a0 * 7, a4 = a0 * 11, a5 = a0 * 13, a6 = a0 * 17, a7 = a0 * 19;
    uint32_t m = seed | 1;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            a0 = a0 * m + a1;
            a1 = a1 * m + a2;
            a2 = a2 * m + a3;
            a3 = a3 * m + a4;
            a4 = a4 * m + a5;
            a5 = a5 * m + a6;
            a6 = a6 * m + a7;
            a7 = a7 * m + a0;
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
}
__global__ void mb_imad_wide(uint64_t* out, uint32_t seed, int iters) {
    // 8 chains of (lo, hi) accumulators: acc_k += lo(acc_{k+1}) * m, written as the same
    // mad.lo.cc / madc.hi pairs the field kernels use (ptxas fuses each pair into one IMAD.WIDE.U32)
    uint32_t l0 = seed + threadIdx.x, l1 = l0 * 3, l2 = l0 * 5, l3 = l0 * 7, l4 = l0 * 11, l5 = l0 * 13, l6 = l0 * 17, l7 = l0 * 19;
    uint32_t h0 = 1, h1 = 2, h2 = 3, h3 = 4, h4 = 5, h5 = 6, h6 = 7, h7 = 8;
    uint32_t m = seed | 1;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            asm volatile(
                "mad.lo.cc.u32 %0, %2, %16, %0;\n\t"
                "madc.hi.u32 %1, %2, %16, %1;\n\t"
                "mad.lo.cc.u32 %2, %4, %16, %2;\n\t"
                "madc.hi.u32 %3, %4, %16, %3;\n\t"
                "mad.lo.cc.u32 %4, %6, %16, %4;\n\t"
                "madc.hi.u32 %5, %6, %16, %5;\n\t"
                "mad.lo.cc.u32 %6, %8, %16, %6;\n\t"
                "madc.hi.u32 %7, %8, %16, %7;\n\t"
                "mad.lo.cc.u32 %8, %10, %16, %8;\n\t"
                "madc.hi.u32 %9, %10, %16, %9;\n\t"
                "mad.lo.cc.u32 %10, %12, %16, %10;\n\t"
                "madc.hi.u32 %11, %12, %16, %11;\n\t"
                "mad.lo.cc.u32 %12, %14, %16, %12;\n\t"
                "madc.hi.u32 %13, %14, %16, %13;\n\t"
                "mad.lo.cc.u32 %14, %0, %16, %14;\n\t"
                "madc.hi.u32 %15, %0, %16, %15;\n\t"
                : "+r"(l0), "+r"(h0), "+r"(l1), "+r"(h1), "+r"(l2), "+r"(h2), "+r"(l3), "+r"(h3), "+r"(l4), "+r"(h4), "+r"(l5), "+r"(h5), "+r"(l6), "+r"(h6), "+r"(l7), "+r"(h7)
                : "r"(m));
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = ((uint64_t)(h0 ^ h1 ^ h2 ^ h3 ^ h4 ^ h5 ^ h6 ^ h7) << 32) | (l0 ^ l1 ^ l2 ^ l3 ^ l4 ^ l5 ^ l6 ^ l7);
}
template <class F>
__global__ void mb_field_mul(F* out, uint32_t seed, int iters) {
    F x = F::from_u32(seed + threadIdx.x), y = F::from_u32(seed * 7 + blockIdx.x), z = x + y, w = x - y;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
        x = x * y;
        y = y * z;
        z = z * w;
        w = w * x;
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = x + y + z + w;
}
__global__ void mb_g1_madd(G1* out, const G1Affine* pts, uint32_t npts, int iters) {
    uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    G1 acc = G1::from_affine(pts[tid % npts]);
    acc = g1_dbl(acc);
#pragma unroll 1
    for (int i = 0; i < iters; i++) g1_madd(acc, pts[(tid + 1 + i) % npts]);
    out[tid] = acc;
}
// FP64 pipe next to the int32 pipe: 8 independent DFMA chains, and the same interleaved with 8 IMAD chains in one thread
__global__ void mb_dfma(double* out, uint32_t seed, int iters) {
    double a0 = seed + threadIdx.x, a1 = a0 * 3, a2 = a0 * 5, a3 = a0 * 7, a4 = a0 * 11, a5 = a0 * 13, a6 = a0 * 17, a7 = a0 * 19;
    const double m = 1.0000001;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            a0 = fma(a0, m, a1);
            a1 = fma(a1, m, a2);
            a2 = fma(a2, m, a3);
            a3 = fma(a3, m, a4);
            a4 = fma(a4, m, a5);
            a5 = fma(a5, m, a6);
            a6 = fma(a6, m, a7);
            a7 = fma(a7, m, a0);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}
__global__ void mb_imad_dfma(double* out, uint32_t seed, int iters) {
    double a0 = seed + threadIdx.x, a1 = a0 * 3, a2 = a0 * 5, a3 = a0 * 7;
    uint32_t b0 = seed + threadIdx.x, b1 = b0 * 3, b2 = b0 * 5, b3 = b0 * 7, b4 = b0 * 11, b5 = b0 * 13, b6 = b0 * 17, b7 = b0 * 19;
    const double m = 1.0000001;
    const uint32_t mi = seed | 1;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            // 8 IMAD + 4 DFMA per round: the issue port is shared, the pipes are not
            b0 = b0 * mi + b1;
            a0 = fma(a0, m, a1);
            b1 = b1 * mi + b2;
            b2 = b2 * mi + b3;
            a1 = fma(a1, m, a2);
            b3 = b3 * mi + b4;
            b4 = b4 * mi + b5;
            a2 = fma(a2, m, a3);
            b5 = b5 * mi + b6;
            b6 = b6 * mi + b7;
            a3 = fma(a3, m, a0);
            b7 = b7 * mi + b0;
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + (double)(b0 ^ b1 ^ b2 ^ b3 ^ b4 ^ b5 ^ b6 ^ b7);
}
// latency of ONE dependent chain per thread (what the one-thread-per-item kernels are bound by): x <- x * x
template <class F>
__global__ void mb_field_chain(F* out, uint32_t seed, int iters) {
    F x = F::one();
    x.v[0] ^= seed + threadIdx.x;
#pragma unroll 1
    for (int i = 0; i < iters; i++) x = x.sqr();
    out[blockIdx.x * blockDim.x + threadIdx.x] = x;
}
// squaring throughput: 4 independent chains per thread, like mb_field_mul
template <class F>
__global__ void mb_field_sqr(F* out, uint32_t seed, int iters) {
    F a = F::one(), b = F::one(), c = F::one(), d = F::one();
    a.v[0] ^= seed + threadIdx.x;
    b.v[1] ^= seed * 3 + threadIdx.x;
    c.v[2] ^= seed * 5 + threadIdx.x;
    d.v[3] ^= seed * 7 + threadIdx.x;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
        a = a.sqr();
        b = b.sqr();
        c = c.sqr();
        d = d.sqr();
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a + b + c + d;
}
template <class F>
__global__ void mb_field_inv(F* out, uint32_t seed, int iters) {
    F x = F::one();
    x.v[0] ^= seed + threadIdx.x;
#pragma unroll 1
    for (int i = 0; i < iters; i++) x = x.inv() + F::one();
    out[blockIdx.x * blockDim.x + threadIdx.x] = x;
}
#endif

}  // namespace dr

using namespace dr;

extern "C" {

// field: 0 = Fq (48-byte big-endian), 1 = Fr, 2 = Fn (32-byte little-endian).  op: 0 mul, 1 add, 2 sub,
// 3 inv(a), 4 sqr(a), 5 neg(a).  Inputs must be canonical.
int dr_field_op(dr_ctx* c, int field, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t count) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || !a || !b || !out || field < 0 || field > 2 || op < 0 || op > 5) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (!count) return DR_OK;
    uint32_t blocks = (uint32_t)((count + 127) / 128);
    if (field == 0) {
        std::vector<Fq> ha(count), hb(count), ho(count);
        for (size_t i = 0; i < count; i++) {
            fq_from_be_bytes_raw(ha[i], a + 48 * i);
            fq_from_be_bytes_raw(hb[i], b + 48 * i);
            if (!ha[i].is_canonical_raw() || !hb[i].is_canonical_raw()) throw Error(DR_EINVAL, "operand is not canonical");
        }
        DevBuf<Fq> da(count), db(count), dout(count);
        h2d(ctx->stream, da.p, ha.data(), count * sizeof(Fq));
        h2d(ctx->stream, db.p, hb.data(), count * sizeof(Fq));
        launch(ctx->stream, Dim3(blocks), 128, 0, FieldOpBody<Fq>(), op, (const Fq*)da.p, (const Fq*)db.p, dout.p, (uint32_t)count);
        d2h(ctx->stream, ho.data(), dout.p, count * sizeof(Fq));
        stream_sync(ctx->stream);
        for (size_t i = 0; i < count; i++) fq_to_be_bytes_raw(out + 48 * i, ho[i]);
    } else {
        std::vector<Fr> ha(count), hb(count), ho(count);
        for (size_t i = 0; i < count; i++) {
            fr_from_le_bytes_raw(ha[i], a + 32 * i);
            fr_from_le_bytes_raw(hb[i], b + 32 * i);
        }
        DevBuf<Fr> da(count), db(count), dout(count);
        h2d(ctx->stream, da.p, ha.data(), count * sizeof(Fr));
        h2d(ctx->stream, db.p, hb.data(), count * sizeof(Fr));
        if (field == 1)
            launch(ctx->stream, Dim3(blocks), 128, 0, FieldOpBody<Fr>(), op, (const Fr*)da.p, (const Fr*)db.p, dout.p, (uint32_t)count);
        else
            launch(ctx->stream, Dim3(blocks), 128, 0, FieldOpBody<Fn>(), op, (const Fn*)da.p, (const Fn*)db.p, (Fn*)dout.p, (uint32_t)count);
        d2h(ctx->stream, ho.data(), dout.p, count * sizeof(Fr));
        stream_sync(ctx->stream);
        for (size_t i = 0; i < count; i++) fr_to_le_bytes_raw(out + 32 * i, ho[i]);
    }
    DR_API_END
}

// kind: 0 IMAD (32-bit mad.lo), 1 IMAD.WIDE (32x32+64), 2 Fq mul, 3 Fr mul, 4 G1 mixed add, 5 DFMA, 6 IMAD + DFMA interleaved (2 : 1),
// 7 / 8 one dependent Fr / Fq squaring chain per warp, one warp per SM (latency), 9 / 10 the same for Fr / Fq inversions,
// 11 / 12 Fq / Fr squaring throughput.
// Returns operations per second over the whole chip and the elapsed ms.
int dr_microbench(dr_ctx* c, int kind, int iters, double* ops_per_s, float* ms_out) {
#if defined(DR_HOST_EMULATION)
    (void)c; (void)kind; (void)iters; (void)ops_per_s; (void)ms_out;
    return set_error(DR_ESTATE, "micro-benchmarks need the CUDA build");
#else
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || iters <= 0 || !ops_per_s) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    cudaDeviceProp prop;
    DR_CUDA(cudaGetDeviceProperties(&prop, ctx->device));
    // kinds 7..10 measure latency: one warp per SM, so nothing hides the dependent chain
    const bool latency = kind >= 7 && kind <= 10;
    const int threads = latency ? 32 : 256;
    const int blocks = prop.multiProcessorCount * (latency ? 1 : (kind >= 2 && kind <= 4) || kind >= 11 ? 2 : 8);
    size_t nthreads = (size_t)blocks * threads;
    DevBuf<uint8_t> out(nthreads * sizeof(G1));
    DevBuf<G1Affine> pts;
    if (kind == 4) {
        // a few hundred distinct multiples of the generator as operands
        std::vector<G1Affine> h(256);
        uint8_t gen[96] = {0x17, 0xf1, 0xd3, 0xa7, 0x31, 0x97, 0xd7, 0x94, 0x26, 0x95, 0x63, 0x8c, 0x4f, 0xa9, 0xac, 0x0f, 0xc3, 0x68, 0x8c, 0x4f, 0x97, 0x74, 0xb9, 0x05,
                           0xa1, 0x4e, 0x3a, 0x3f, 0x17, 0x1b, 0xac, 0x58, 0x6c, 0x55, 0xe8, 0x3f, 0xf9, 0x7a, 0x1a, 0xef, 0xfb, 0x3a, 0xf0, 0x0a, 0xdb, 0x22, 0xc6, 0xbb,
                           0x08, 0xb3, 0xf4, 0x81, 0xe3, 0xaa, 0xa0, 0xf1, 0xa0, 0x9e, 0x30, 0xed, 0x74, 0x1d, 0x8a, 0xe4, 0xfc, 0xf5, 0xe0, 0x95, 0xd5, 0xd0, 0x0a, 0xf6,
                           0x00, 0xdb, 0x18, 0xcb, 0x2c, 0x04, 0xb3, 0xed, 0xd0, 0x3c, 0xc7, 0x44, 0xa2, 0x88, 0x8a, 0xe4, 0x0c, 0xaa, 0x23, 0x29, 0x46, 0xc5, 0xe7, 0xe1};
        G1Affine g;
        if (!g1_decode(g, gen, 96)) throw Error(DR_ESTATE, "generator decode failed");
        G1 acc = G1::from_affine(g);
        for (auto& p : h) {
            acc = g1_dbl(acc);
            g1_madd(acc, g);
            p = g1_to_affine(acc);
        }
        pts.alloc(h.size());
        h2d(ctx->stream, pts.p, h.data(), h.size() * sizeof(G1Affine));
    }
    double per_thread = 0;
    for (int rep = 0; rep < 2; rep++) {  // first repetition warms up
        dr_ctx_timer_start(c);
        switch (kind) {
            case 0: mb_imad32<<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out.p, 12345u, iters); per_thread = 64.0 * iters; break;
            case 1: mb_imad_wide<<<blocks, threads, 0, ctx->stream>>>((uint64_t*)out.p, 12345u, iters); per_thread = 64.0 * iters; break;
            case 2: mb_field_mul<Fq><<<blocks, threads, 0, ctx->stream>>>((Fq*)out.p, 12345u, iters); per_thread = 4.0 * iters; break;
            case 3: mb_field_mul<Fr><<<blocks, threads, 0, ctx->stream>>>((Fr*)out.p, 12345u, iters); per_thread = 4.0 * iters; break;
            case 4: mb_g1_madd<<<blocks, threads, 0, ctx->stream>>>((G1*)out.p, pts.p, 256u, iters); per_thread = 1.0 * iters; break;
            case 5: mb_dfma<<<blocks, threads, 0, ctx->stream>>>((double*)out.p, 12345u, iters); per_thread = 64.0 * iters; break;
            case 6: mb_imad_dfma<<<blocks, threads, 0, ctx->stream>>>((double*)out.p, 12345u, iters); per_thread = 96.0 * iters; break;  // 64 IMAD + 32 DFMA
            case 7: mb_field_chain<Fr><<<blocks, threads, 0, ctx->stream>>>((Fr*)out.p, 12345u, iters); per_thread = 1.0 * iters; break;
            case 8: mb_field_chain<Fq><<<blocks, threads, 0, ctx->stream>>>((Fq*)out.p, 12345u, iters); per_thread = 1.0 * iters; break;
            case 9: mb_field_inv<Fr><<<blocks, threads, 0, ctx->stream>>>((Fr*)out.p, 12345u, iters); per_thread = 1.0 * iters; break;
            case 10: mb_field_inv<Fq><<<blocks, threads, 0, ctx->stream>>>((Fq*)out.p, 12345u, iters); per_thread = 1.0 * iters; break;
            case 11: mb_field_sqr<Fq><<<blocks, threads, 0, ctx->stream>>>((Fq*)out.p, 12345u, iters); per_thread = 4.0 * iters; break;
            case 12: mb_field_sqr<Fr><<<blocks, threads, 0, ctx->stream>>>((Fr*)out.p, 12345u, iters); per_thread = 4.0 * iters; break;
            default: throw Error(DR_EINVAL, "unknown micro-benchmark");
        }
        DR_CUDA(cudaGetLastError());
        launch_counter()++;
        float ms = 0;
        dr_ctx_timer_stop(c, &ms);
        if (ms_out) *ms_out = ms;
        *ops_per_s = per_thread * (double)nthreads / (ms * 1e-3);
    }
    DR_API_END
#endif
}
}
