// C ABI, part 1: context, SRS + fixed-base table, KZG commit, G1 codecs, Fr NTT.
#include "api_internal.cuh"

namespace dr {

thread_local std::string g_last_error;

int set_error(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

// ---- fixed-base tables for Bandersnatch scalar multiplications (te.cuh: te_mul_fixed) ----------------
std::shared_ptr<Ctx::FixedTable> Ctx::fixed_table(const TEAffine& base) {
    for (auto& t : fixed_tables)
        if (t->base == base) return t;
    auto t = std::make_shared<FixedTable>();
    t->base = base;
    t->tab.alloc(TE_FIXED_ENTRIES);
    launch(stream, Dim3(TE_FIXED_WINDOWS * 16 / 32), 32, 0, TeFixedTableBody(), base, t->tab.p);
    stream_sync(stream);
    if (fixed_tables.size() >= FIXED_TABLE_CAP) fixed_tables.erase(fixed_tables.begin());
    fixed_tables.push_back(t);
    return t;
}

// ---- NTT plans (twiddle tables per (n, omega)) -----------------------------------------------------
const NttPlan& Ctx::plan(uint32_t n, const Fr& omega_mont) {
    for (auto& p : plans)
        if (p->n == n && p->omega == omega_mont) return *p;
    auto p = std::make_unique<NttPlan>();
    p->n = n;
    p->logn = 0;
    while ((1u << p->logn) < n) p->logn++;
    p->omega = omega_mont;
    Fr omega_inv = omega_mont.inv();
    Fr ninv = Fr::from_u32(n).inv();
    p->n_inv.alloc(1);
    h2d(stream, p->n_inv.p, &ninv, sizeof(Fr));
    if (n <= 4096) {
        std::vector<Fr> fwd(n / 2 ? n / 2 : 1), inv(n / 2 ? n / 2 : 1);
        Fr w = Fr::one(), wi = Fr::one();
        for (uint32_t k = 0; k < n / 2; k++) {
            fwd[k] = w;
            inv[k] = wi;
            w = w * omega_mont;
            wi = wi * omega_inv;
        }
        p->tw_fwd.alloc(fwd.size());
        p->tw_inv.alloc(inv.size());
        h2d(stream, p->tw_fwd.p, fwd.data(), fwd.size() * sizeof(Fr));
        h2d(stream, p->tw_inv.p, inv.data(), inv.size() * sizeof(Fr));
        stream_sync(stream);
    } else {
        p->logn1 = (p->logn + 1) / 2;
        p->logn2 = p->logn - p->logn1;
        p->n1 = 1u << p->logn1;
        p->n2 = 1u << p->logn2;
        for (int dir = 0; dir < 2; dir++) {
            const Fr base = dir ? omega_inv : omega_mont;
            std::vector<Fr> full(n), t1(p->n1 / 2), t2(p->n2 / 2);
            Fr w = Fr::one();
            for (uint32_t i = 0; i < n; i++) {
                full[i] = w;
                w = w * base;
            }
            for (uint32_t k = 0; k < p->n1 / 2; k++) t1[k] = full[(size_t)k * p->n2];  // (w^n2)^k
            for (uint32_t k = 0; k < p->n2 / 2; k++) t2[k] = full[(size_t)k * p->n1];  // (w^n1)^k
            p->wfull[dir].alloc(n);
            p->tw1[dir].alloc(t1.size());
            p->tw2[dir].alloc(t2.size());
            h2d(stream, p->wfull[dir].p, full.data(), (size_t)n * sizeof(Fr));
            h2d(stream, p->tw1[dir].p, t1.data(), t1.size() * sizeof(Fr));
            h2d(stream, p->tw2[dir].p, t2.data(), t2.size() * sizeof(Fr));
            stream_sync(stream);
        }
    }
    plans.push_back(std::move(p));
    return *plans.back();
}

void ntt_device(Ctx* ctx, const NttPlan& plan, const Fr* in, Fr* out, size_t batch, bool inverse, DevBuf<Fr>& tmp) {
    const uint32_t n = plan.n;
    if (n <= 4096) {
        const uint32_t threads = ntt_threads(n);
        launch(ctx->stream, Dim3((uint32_t)batch), threads, ntt_smem_bytes(n), NttPlainBody(), in, out, n, plan.logn, (const Fr*)(inverse ? plan.tw_inv.p : plan.tw_fwd.p),
               (const Fr*)(inverse ? plan.n_inv.p : nullptr));
        return;
    }
    const int dir = inverse ? 1 : 0;
    tmp.ensure((size_t)n * batch);
    launch(ctx->stream, Dim3(plan.n2, (uint32_t)batch), ntt_threads(plan.n1), ntt_smem_bytes(plan.n1), NttLargePass1Body(), in, tmp.p, plan.n1, plan.logn1, plan.n2, (const Fr*)plan.tw1[dir].p,
           (const Fr*)plan.wfull[dir].p);
    launch(ctx->stream, Dim3(plan.n1, (uint32_t)batch), ntt_threads(plan.n2), ntt_smem_bytes(plan.n2), NttLargePass2Body(), (const Fr*)tmp.p, out, plan.n1, plan.n2, plan.logn2,
           (const Fr*)plan.tw2[dir].p, (const Fr*)(inverse ? plan.n_inv.p : nullptr));
}

void PhaseTimer::mark(Ctx* ctx, int phase) {
    size_t i = phase_of.size();
    phase_of.push_back(phase);
    if (phase != 6 && phase < 7) current = phase;
#if !defined(DR_HOST_EMULATION)
    if (events.size() <= i) {
        cudaEvent_t e;
        DR_CUDA(cudaEventCreate(&e));
        events.push_back(e);
    }
    DR_CUDA(cudaEventRecord(events[i], ctx->stream));
#else
    (void)ctx;
    if (stamps.size() <= i) stamps.resize(i + 1);
    stamps[i] = std::chrono::steady_clock::now();
#endif
}

int PhaseTimer::current_of(size_t i) const {
    while (i > 0) {
        i--;
        if (phase_of[i] != 6) return phase_of[i] >= 0 && phase_of[i] < 6 ? phase_of[i] : 5;
    }
    return 5;
}

void PhaseTimer::collect(Ctx* ctx) {
    (void)ctx;
    for (size_t i = 0; i + 1 < phase_of.size(); i++) {
        int ph = phase_of[i];
        if (ph < 0 || ph >= NPH) continue;
        float ms = 0;
#if !defined(DR_HOST_EMULATION)
        DR_CUDA(cudaEventElapsedTime(&ms, events[i], events[i + 1]));
#else
        ms = std::chrono::duration<float, std::milli>(stamps[i + 1] - stamps[i]).count();
#endif
        total[ph] += ms;
        if (ph == 6) total[current_of(i)] += ms;  // the kernel-only span is part of its enclosing phase
    }
    phase_of.clear();
}

void build_window_table(Ctx* ctx, const G1Affine* points, const TableGeom& geom, DevBuf<G1Affine>& table) {
    if (geom.W > 64) throw Error(DR_EINVAL, "window_bits too small");
    table.alloc(geom.total_entries());
    uint32_t chunks = geom.max_entries() >= 512 ? (geom.max_entries() + 255) / 256 : 1;  // <= 256 serial additions per thread
    const uint32_t maxw = geom.W <= 32 ? 32 : 64, runs = maxw / geom.W;  // TableBuildBody: runs of 256 digits per thread
    size_t nthreads = (size_t)geom.n_points * ((chunks + runs - 1) / runs);
    const uint32_t tb = 64;
    Dim3 grid((uint32_t)((nthreads + tb - 1) / tb));
    if (geom.W <= 32)
        launch(ctx->stream, grid, tb, 0, TableBuildBody<32>(), points, table.p, geom, chunks);
    else
        launch(ctx->stream, grid, tb, 0, TableBuildBody<64>(), points, table.p, geom, chunks);
}

const LagrangeTable& Srs::lagrange_table(uint32_t N, uint32_t logN, const Fr& omega, const Fr* tw_inv_half, const Fr& n_inv) {
    for (auto& l : lagrange)
        if (l->N == N && l->omega == omega) return *l;
    if (N > n) throw Error(DR_EINVAL, "SRS smaller than the domain");
    auto l = std::make_unique<LagrangeTable>();
    l->N = N;
    l->omega = omega;
    DevBuf<G1> work(N);
    DevBuf<G1Affine> sj(N);
    Stream st = ctx->stream;
    launch(st, Dim3((N + 63) / 64), 64, 0, G1BitReverseBody(), (const G1Affine*)points.p, N, logN, work.p);
    for (uint32_t half = 1; half < N; half <<= 1) launch(st, Dim3((N / 2 + 31) / 32), 32, 0, G1NttStageBody(), work.p, N, half, tw_inv_half);
    launch(st, Dim3((N + 31) / 32), 32, 0, G1ScaleBody(), work.p, N, n_inv);
    const uint32_t pt = 128;
    launch(st, Dim3(1), pt, pt * sizeof(G1), G1PrefixSumBody(), work.p, N, sj.p);
    // 10-bit windows: 2.6 GB at N = 2048, 26 additions per step (12 bits = 8.9 GB and 22 additions were measured: the commit phase
    // gains 0.5 %, not worth the memory); follows a smaller SRS window (tests)
    const uint32_t lc = geom.c < 10 ? geom.c : 10;
    l->geom = make_geom(lc, N);
    build_window_table(ctx, sj.p, l->geom, l->table);
    stream_sync(st);
    lagrange.push_back(std::move(l));
    return *lagrange.back();
}

#ifndef DR_COMMIT_MINB
#define DR_COMMIT_MINB 4
#endif

// Slices per polynomial: the grid is (slices, batch) CTAs of which 4 are resident per SM, so batch * slices should fill a whole
// number of waves -- a 2.6-wave grid runs as long as a 3-wave one (measured: 512 proofs x 3 slices cost 13 % more per proof
// than 4096 x 1, which happens to be 6.92 waves).  Among the splits that keep >= 32 points per CTA take the one with the best
// wave occupancy, smaller splits first (every CTA ends in a 7-level reduction tree).
static uint32_t commit_slices(Ctx* ctx, uint32_t n, uint32_t batch) {
    uint32_t slices = 1;
    const uint32_t resident = ctx->sm_count() * DR_COMMIT_MINB;
    const uint32_t finest = n / 32 ? n / 32 : 1;  // >= 32 points per CTA
    if ((uint64_t)batch * finest <= resident) return finest;  // not even one wave: as many CTAs as the polynomial allows (single proofs, small batches)
    const uint32_t max_slices = finest < 256 ? finest : 256;
    double best = -1.0;
    for (uint32_t s = 1; s <= max_slices; s++) {
        const double waves = (double)batch * s / resident;
        const double whole = (double)(uint64_t)(waves + 0.999999);
        const double score = (waves < 1.0 ? waves : waves / whole) - 0.004 * s;
        if (score > best + 1e-9) {
            best = score;
            slices = s;
        }
    }
    return slices;
}

// the dense commit kernel alone: partials[b * slices + s] = XYZZ sum of slice s of polynomial b
// partial sums a CTA of the dense commit kernel leaves for the finish kernel (see CommitBodyT)
// (only for moderately sliced launches: with hundreds of slices per polynomial -- a single proof -- the finish kernel's lanes would
// fold hundreds of partial sums each)
static uint32_t commit_keep(uint32_t slices) { return slices > 1 && slices <= 16 ? 32u : 1u; }

static void commit_launch(Ctx* ctx, Srs* srs, const Fr* scalars, size_t stride, uint32_t n, uint32_t batch, uint32_t slices, G1* partials) {
    const uint32_t keep = commit_keep(slices);
    const uint32_t threads = COMMIT_THREADS;
    PhaseTimer& pt = ctx->phases;
    const int enclosing = pt.current;
    if (pt.active) {
        pt.mark(ctx, 6);
        pt.kernel_launches++;
    }
    if (srs->geom.glv)
        launch_lb<COMMIT_THREADS, DR_COMMIT_MINB>(ctx->stream, Dim3(slices, batch), threads, threads * sizeof(G1), CommitGlvBody(), (const G1Affine*)srs->table.p, srs->geom, scalars, stride, n, partials, keep);
    else
        launch_lb<COMMIT_THREADS, DR_COMMIT_MINB>(ctx->stream, Dim3(slices, batch), threads, threads * sizeof(G1), CommitBody(), (const G1Affine*)srs->table.p, srs->geom, scalars, stride, n, partials, keep);
    if (pt.active) pt.mark(ctx, enclosing);
}

void commit_device(Ctx* ctx, Srs* srs, const Fr* scalars, size_t stride, uint32_t n, uint32_t batch, G1Affine* out_affine) {
    if (n == 0 || batch == 0) return;
    if (n > srs->n) throw Error(DR_EINVAL, "polynomial degree exceeds SRS size");
    if (ctx->commit_mode == 1 && !srs->geom.glv && ((size_t)(n + 31) / 32) * srs->geom.W >= 2 * AFFINE_MIN_PAIRS) {
        // batched-affine rounds: one warp per (polynomial, slice), persistent CTAs of 4 warps, HBM scratch per resident lane
        const uint32_t warps = COMMIT_THREADS / 32;
        const uint32_t resident = 148 * 4;
        // slices: enough warps to fill the machine, while a lane keeps >= 4 rounds' worth of references
        uint32_t slices = 1;
        while (batch * slices < resident * warps && ((size_t)(n + 32 * slices * 2 - 1) / (32 * slices * 2)) * srs->geom.W >= 8 * AFFINE_MIN_PAIRS) slices *= 2;
        const uint32_t items = batch * slices;
        uint32_t ctas = (items + warps - 1) / warps;
        if (ctas > resident) ctas = resident;
        const uint32_t slots = ctas * warps;
        uint32_t cap = ((n + 32 * slices - 1) / (32 * slices)) * srs->geom.W;
        cap = (cap + 3) & ~3u;
        ctx->aff_refs.ensure((size_t)slots * cap * 32);
        ctx->aff_prefix.ensure((size_t)slots * (cap / 2) * 32);
        ctx->aff_a.ensure((size_t)slots * (cap / 2) * 32);
        ctx->aff_b.ensure((size_t)slots * (cap / 4) * 32);
        AffineScratch sc{ctx->aff_refs.p, ctx->aff_prefix.p, ctx->aff_a.p, ctx->aff_b.p, cap};
        ctx->partials.ensure(items);
        launch_lb<COMMIT_THREADS, DR_COMMIT_MINB>(ctx->stream, Dim3(ctas), COMMIT_THREADS, COMMIT_THREADS * sizeof(G1), CommitAffineBody(), (const G1Affine*)srs->table.p,
                                                  srs->geom, scalars, stride, n, batch, slices, sc, ctx->partials.p);
        launch_commit_finish(ctx->stream, (const G1*)ctx->partials.p, slices, batch, out_affine);
        return;
    }
    const uint32_t slices = commit_slices(ctx, n, batch), keep = commit_keep(slices);
    ctx->partials.ensure((size_t)batch * slices * keep);
    commit_launch(ctx, srs, scalars, stride, n, batch, slices, ctx->partials.p);
    launch_commit_finish(ctx->stream, (const G1*)ctx->partials.p, slices * keep, batch, out_affine);
}

// Two commitments of the same batch whose results nothing needs in between (the prover's two opening proofs): both commit kernels,
// then ONE finish launch over 2 * batch sums -- a finish is a latency-bound kernel (one field inversion per sum) and a pass pays
// each of them in full whatever its width.  out_affine: batch results of the first, then batch results of the second.
void commit_device_pair(Ctx* ctx, Srs* srs, const Fr* scalars_a, size_t stride_a, uint32_t n_a, const Fr* scalars_b, size_t stride_b, uint32_t n_b, uint32_t batch,
                        G1Affine* out_affine) {
    const bool plain = !(ctx->commit_mode == 1 && !srs->geom.glv);
    const uint32_t sa = n_a && batch ? commit_slices(ctx, n_a, batch) : 0, sb = n_b && batch ? commit_slices(ctx, n_b, batch) : 0;
    if (!plain || !sa || sa != sb) {
        commit_device(ctx, srs, scalars_a, stride_a, n_a, batch, out_affine);
        commit_device(ctx, srs, scalars_b, stride_b, n_b, batch, out_affine + batch);
        return;
    }
    if (n_a > srs->n || n_b > srs->n) throw Error(DR_EINVAL, "polynomial degree exceeds SRS size");
    const uint32_t keep = commit_keep(sa);
    ctx->partials.ensure((size_t)2 * batch * sa * keep);
    commit_launch(ctx, srs, scalars_a, stride_a, n_a, batch, sa, ctx->partials.p);
    commit_launch(ctx, srs, scalars_b, stride_b, n_b, batch, sa, ctx->partials.p + (size_t)batch * sa * keep);
    launch_commit_finish(ctx->stream, (const G1*)ctx->partials.p, sa * keep, 2 * batch, out_affine);
}

}  // namespace dr

using namespace dr;

#define DR_API_BEGIN try {
#define DR_API_END                                   \
    }                                                \
    catch (const Error& e) {                         \
        return set_error(e.code, e.what());          \
    }                                                \
    catch (const std::exception& e) {                \
        return set_error(DR_ECUDA, e.what());        \
    }                                                \
    return DR_OK;

extern "C" {

const char* dr_last_error(void) { return g_last_error.c_str(); }
const char* dr_version(void) { return "dot_ring_b200 0.1 (sm_100a)"; }
int dr_is_cuda_build(void) {
#if defined(DR_HOST_EMULATION)
    return 0;
#else
    return 1;
#endif
}
uint64_t dr_launch_count(void) { return launch_counter(); }
int dr_device_count(void) {
#if defined(DR_HOST_EMULATION)
    return 1;
#else
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return count;
#endif
}

int dr_ctx_create(int device, dr_ctx** out) {
    DR_API_BEGIN
    if (!out) throw Error(DR_EINVAL, "null out pointer");
    auto ctx = std::make_unique<Ctx>();
    ctx->device = device;
#if !defined(DR_HOST_EMULATION)
    int count = 0;
    DR_CUDA(cudaGetDeviceCount(&count));
    if (device < 0 || device >= count) throw Error(DR_EINVAL, "no such CUDA device");
    DR_CUDA(cudaSetDevice(device));
    DR_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    DR_CUDA(cudaStreamCreateWithFlags(&ctx->side, cudaStreamNonBlocking));
    DR_CUDA(cudaStreamCreateWithFlags(&ctx->side2, cudaStreamNonBlocking));
    DR_CUDA(cudaEventCreateWithFlags(&ctx->ev_fork2, cudaEventDisableTiming));
    DR_CUDA(cudaEventCreateWithFlags(&ctx->ev_join2, cudaEventDisableTiming));
    DR_CUDA(cudaEventCreate(&ctx->ev_fork));
    DR_CUDA(cudaEventCreate(&ctx->ev_join));
    // Fix the per-thread stack once: kernels here need between 0 and ~16 KB of local memory, and letting the runtime grow the
    // backing store lazily costs a device-wide reallocation (hundreds of ms) whenever a larger kernel follows a smaller one.
    if (const char* e = getenv("DOT_RING_B200_STACK_BYTES")) {
        DR_CUDA(cudaDeviceSetLimit(cudaLimitStackSize, (size_t)atol(e)));
    } else {
        DR_CUDA(cudaDeviceSetLimit(cudaLimitStackSize, 16 * 1024));
    }
    DR_CUDA(cudaEventCreate(&ctx->ev_start));
    DR_CUDA(cudaEventCreate(&ctx->ev_stop));
#else
    ctx->stream = 0;
    ctx->side = 0;
    ctx->side2 = 0;
#endif
    {
        std::lock_guard<std::mutex> lock(live_ctx_mutex());
        live_ctxs().insert(ctx.get());
    }
    *out = (dr_ctx*)ctx.release();
    DR_API_END
}

void dr_ctx_destroy(dr_ctx* c) {
    Ctx* ctx = (Ctx*)c;
    if (!ctx) return;
    {
        std::lock_guard<std::mutex> lock(live_ctx_mutex());
        live_ctxs().erase(ctx);
    }
#if !defined(DR_HOST_EMULATION)
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->side);
    cudaStreamSynchronize(ctx->side2);
    current_stream() = ctx->stream;
#endif
    ctx->plans.clear();
    ctx->release_scratch();
#if !defined(DR_HOST_EMULATION)
    cudaEventDestroy(ctx->ev_start);
    cudaEventDestroy(ctx->ev_stop);
    cudaEventDestroy(ctx->ev_fork);
    cudaEventDestroy(ctx->ev_join);
    cudaEventDestroy(ctx->ev_fork2);
    cudaEventDestroy(ctx->ev_join2);
    cudaStreamDestroy(ctx->side2);
    cudaStreamDestroy(ctx->side);
    cudaStreamDestroy(ctx->stream);
    current_stream() = nullptr;
#endif
    delete ctx;
}

int dr_ctx_set_commit_mode(dr_ctx* c, int mode) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || mode < 0 || mode > 1) throw Error(DR_EINVAL, "bad argument");
    ctx->commit_mode = mode;
    DR_API_END
}

int dr_ctx_trim(dr_ctx* c) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    stream_sync(ctx->stream);
#if !defined(DR_HOST_EMULATION)
    dev_cache_trim();
#endif
    DR_API_END
}

int dr_ctx_sync(dr_ctx* c) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    ctx->activate();
    stream_sync(ctx->stream);
    DR_API_END
}

int dr_ctx_timer_start(dr_ctx* c) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    ctx->activate();
#if !defined(DR_HOST_EMULATION)
    DR_CUDA(cudaEventRecord(ctx->ev_start, ctx->stream));
#else
    ctx->t_start = std::chrono::steady_clock::now();
#endif
    DR_API_END
}

int dr_ctx_timer_stop(dr_ctx* c, float* ms_out) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    ctx->activate();
#if !defined(DR_HOST_EMULATION)
    DR_CUDA(cudaEventRecord(ctx->ev_stop, ctx->stream));
    DR_CUDA(cudaEventSynchronize(ctx->ev_stop));
    DR_CUDA(cudaEventElapsedTime(ms_out, ctx->ev_start, ctx->ev_stop));
#else
    *ms_out = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - ctx->t_start).count();
#endif
    DR_API_END
}

int dr_ctx_device_info(dr_ctx* c, char* name_buf, size_t name_len, int* sm_count, int* sm_clock_khz, size_t* free_bytes, size_t* total_bytes) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    ctx->activate();
#if !defined(DR_HOST_EMULATION)
    cudaDeviceProp prop;
    DR_CUDA(cudaGetDeviceProperties(&prop, ctx->device));
    if (name_buf && name_len) snprintf(name_buf, name_len, "%s", prop.name);
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (sm_clock_khz) {
        int khz = 0;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
        *sm_clock_khz = khz;
    }
    size_t f = 0, t = 0;
    DR_CUDA(cudaMemGetInfo(&f, &t));
    if (free_bytes) *free_bytes = f;
    if (total_bytes) *total_bytes = t;
#else
    if (name_buf && name_len) snprintf(name_buf, name_len, "cpu-emulation");
    if (sm_count) *sm_count = 0;
    if (sm_clock_khz) *sm_clock_khz = 0;
    if (free_bytes) *free_bytes = 0;
    if (total_bytes) *total_bytes = 0;
#endif
    DR_API_END
}

// ---------------------------------------------------------------------------------------- SRS
int dr_srs_load(dr_ctx* c, const uint8_t* g1_be96, size_t n_g1, const uint8_t* g2_be192, int window_bits, dr_srs** out) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || !g1_be96 || !g2_be192 || !out || n_g1 == 0) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    uint32_t cbits = (uint32_t)window_bits & 0xff, wide = ((uint32_t)window_bits >> 8) & 0xff, glv = ((uint32_t)window_bits >> 16) & 1;
    if (window_bits <= 0) {
        // the table with the fewest additions per coefficient that the free device memory can hold next to the prover's scratch
        cbits = 8;
        wide = 0;
#if !defined(DR_HOST_EMULATION)
        size_t free_b = 0, total_b = 0;
        DR_CUDA(cudaMemGetInfo(&free_b, &total_b));
        free_b += dev_cache().cached;
        auto fits = [&](uint32_t c, uint32_t k) {
            size_t bytes = make_geom(c, (uint32_t)n_g1, k).total_entries() * sizeof(G1Affine);
            size_t reserve = bytes / 4 > ((size_t)24 << 30) ? bytes / 4 : ((size_t)24 << 30);
            return bytes + reserve <= free_b;
        };
        // first choice on a 180 GB part: 16-bit windows over the GLV halves (16 additions per coefficient, 161 GB for 6145 points),
        // as long as 14 GB stay free next to it: the ring tables (2.6 GB) and a 4096-proof pass (7.5 GB of scratch)
        const size_t glv_bytes = make_geom(16, (uint32_t)n_g1, 0, 1).total_entries() * sizeof(G1Affine);
        if (glv_bytes + ((size_t)14 << 30) <= free_b) {
            cbits = 16;
            wide = 0;
            glv = 1;
        } else if (fits(14, 4)) {
            cbits = 14;
            wide = 4;
        } else {
            for (uint32_t c = 14; c >= 8; c--) {
                if (fits(c, 0)) {
                    cbits = c;
                    break;
                }
            }
        }
#endif
    } else if (window_bits >> 17) {
        throw Error(DR_EINVAL, "bad window_bits");
    }
    if (cbits < 2 || cbits > (glv ? 16u : 15u)) throw Error(DR_EINVAL, "window_bits must be in [2, 15] (16 with the GLV split)");
    if (wide && (cbits + 1 > 16 || wide > make_geom(cbits, 1, wide, glv).W)) throw Error(DR_EINVAL, "bad number of wide windows");
    auto srs = std::make_unique<Srs>();
    srs->ctx = ctx;
    srs->n = (uint32_t)n_g1;
    memcpy(srs->g1_0_be96, g1_be96, 96);
    memcpy(srs->g2_be192, g2_be192, 384);
    srs->geom = make_geom(cbits, srs->n, wide, glv);
    DevBuf<uint8_t> raw(n_g1 * 96);
    DevBuf<uint32_t> bad(1);
    dev_zero(ctx->stream, bad.p, 4);
    h2d(ctx->stream, raw.p, g1_be96, n_g1 * 96);
    srs->points.alloc(n_g1);
    launch(ctx->stream, Dim3((srs->n + 127) / 128), 128, 0, SrsLoadBody(), (const uint8_t*)raw.p, srs->points.p, srs->n, bad.p);
    uint32_t bad_h = 0;
    d2h(ctx->stream, &bad_h, bad.p, 4);
    stream_sync(ctx->stream);
    if (bad_h) throw Error(DR_EINVAL, "invalid BLS12-381 G1 encoding in SRS");
    // fixed-base table
    build_window_table(ctx, srs->points.p, srs->geom, srs->table);
    stream_sync(ctx->stream);
    *out = (dr_srs*)srs.release();
    DR_API_END
}

void dr_srs_destroy(dr_srs* s) {
    Srs* srs = (Srs*)s;
    if (!srs) return;
    free_on_owner_stream(srs->ctx);
    delete srs;
}
size_t dr_srs_size(const dr_srs* s) { return s ? ((const Srs*)s)->n : 0; }
void dr_srs_geometry(const dr_srs* s, uint32_t* window_bits, uint32_t* wide_windows, uint32_t* glv, uint32_t* additions) {
    const TableGeom g = s ? ((const Srs*)s)->geom : TableGeom{};
    if (window_bits) *window_bits = g.c;
    if (wide_windows) *wide_windows = g.wide;
    if (glv) *glv = g.glv;
    if (additions) *additions = s ? g.additions() : 0;
}
size_t dr_srs_table_bytes(const dr_srs* s) { return s ? ((const Srs*)s)->geom.total_entries() * sizeof(G1Affine) : 0; }

int dr_kzg_commit(dr_ctx* c, dr_srs* s, const uint8_t* coeffs_le32, size_t n, size_t batch, uint8_t* out_be96) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    Srs* srs = (Srs*)s;
    if (!ctx || !srs || !out_be96 || (!coeffs_le32 && n * batch)) throw Error(DR_EINVAL, "bad argument");
    if (n > srs->n) throw Error(DR_EINVAL, "polynomial degree exceeds SRS size");
    ctx->activate();
    if (batch == 0) return DR_OK;
    if (n == 0) {  // empty polynomial commits to infinity
        for (size_t b = 0; b < batch; b++) {
            memset(out_be96 + 96 * b, 0, 96);
            out_be96[96 * b] = 0x40;
        }
        return DR_OK;
    }
    size_t total = n * batch;
    DevBuf<uint8_t> raw(total * 32);
    DevBuf<Fr> sc(total);
    DevBuf<G1Affine> res(batch);
    DevBuf<uint8_t> enc(batch * 96);
    h2d(ctx->stream, raw.p, coeffs_le32, total * 32);
    launch(ctx->stream, Dim3((uint32_t)((total + 255) / 256)), 256, 0, FrToMontBody(), (const uint8_t*)raw.p, sc.p, total, (uint32_t*)nullptr);
    commit_device(ctx, srs, sc.p, n, (uint32_t)n, (uint32_t)batch, res.p);
    launch(ctx->stream, Dim3((uint32_t)((batch + 63) / 64)), 64, 0, G1EncodeBody(), (const G1Affine*)res.p, (uint32_t)batch, enc.p, (uint8_t*)nullptr);
    d2h(ctx->stream, out_be96, enc.p, batch * 96);
    stream_sync(ctx->stream);
    DR_API_END
}

// splitmix64-based deterministic scalars generated on the device side of the ABI (host fills, uploads once)
static uint64_t splitmix64(uint64_t& x) {
    uint64_t z = (x += 0x9E3779B97F4A7C15ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

int dr_kzg_commit_bench(dr_ctx* c, dr_srs* s, size_t n, size_t batch, int iters, uint64_t seed, float* ms_per_iter, uint8_t* out_first_be96) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    Srs* srs = (Srs*)s;
    if (!ctx || !srs || n == 0 || batch == 0 || iters <= 0 || n > srs->n) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    size_t total = n * batch;
    std::vector<uint8_t> host(total * 32);
    uint64_t st = seed;
    for (size_t i = 0; i < total; i++) {
        uint64_t w[4] = {splitmix64(st), splitmix64(st), splitmix64(st), splitmix64(st) >> 2};  // < 2^254 < r
        memcpy(&host[32 * i], w, 32);
    }
    DevBuf<uint8_t> raw(total * 32);
    DevBuf<Fr> sc(total);
    DevBuf<G1Affine> res(batch);
    h2d(ctx->stream, raw.p, host.data(), total * 32);
    launch(ctx->stream, Dim3((uint32_t)((total + 255) / 256)), 256, 0, FrToMontBody(), (const uint8_t*)raw.p, sc.p, total, (uint32_t*)nullptr);
    commit_device(ctx, srs, sc.p, n, (uint32_t)n, (uint32_t)batch, res.p);  // warm-up
    stream_sync(ctx->stream);
    float ms = 0;
    dr_ctx_timer_start(c);
    for (int it = 0; it < iters; it++) commit_device(ctx, srs, sc.p, n, (uint32_t)n, (uint32_t)batch, res.p);
    dr_ctx_timer_stop(c, &ms);
    if (ms_per_iter) *ms_per_iter = ms / iters;
    if (out_first_be96) {
        DevBuf<uint8_t> enc(96);
        launch(ctx->stream, Dim3(1), 64, 0, G1EncodeBody(), (const G1Affine*)res.p, 1u, enc.p, (uint8_t*)nullptr);
        d2h(ctx->stream, out_first_be96, enc.p, 96);
        stream_sync(ctx->stream);
    }
    DR_API_END
}

// ------------------------------------------------------------------------------------- G1 codecs
int dr_g1_compress(dr_ctx* c, const uint8_t* in_be96, size_t count, uint8_t* out_be48) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || (count && (!in_be96 || !out_be48))) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (!count) return DR_OK;
    DevBuf<uint8_t> raw(count * 96), ok(count), enc(count * 48);
    DevBuf<G1Affine> pts(count);
    h2d(ctx->stream, raw.p, in_be96, count * 96);
    uint32_t blocks = (uint32_t)((count + 63) / 64);
    launch(ctx->stream, Dim3(blocks), 64, 0, G1DecodeBody(), (const uint8_t*)raw.p, 96u, (uint32_t)count, pts.p, ok.p);
    launch(ctx->stream, Dim3(blocks), 64, 0, G1EncodeBody(), (const G1Affine*)pts.p, (uint32_t)count, (uint8_t*)nullptr, enc.p);
    std::vector<uint8_t> okh(count);
    d2h(ctx->stream, okh.data(), ok.p, count);
    d2h(ctx->stream, out_be48, enc.p, count * 48);
    stream_sync(ctx->stream);
    for (size_t i = 0; i < count; i++)
        if (!okh[i]) throw Error(DR_EINVAL, "invalid BLS12-381 G1 encoding");
    DR_API_END
}

int dr_g1_decompress(dr_ctx* c, const uint8_t* in_be48, size_t count, uint8_t* out_be96, uint8_t* ok_out) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || (count && (!in_be48 || !out_be96 || !ok_out))) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (!count) return DR_OK;
    DevBuf<uint8_t> raw(count * 48), ok(count), enc(count * 96);
    DevBuf<G1Affine> pts(count);
    h2d(ctx->stream, raw.p, in_be48, count * 48);
    uint32_t blocks = (uint32_t)((count + 63) / 64);
    launch(ctx->stream, Dim3(blocks), 64, 0, G1DecodeBody(), (const uint8_t*)raw.p, 48u, (uint32_t)count, pts.p, ok.p);
    launch(ctx->stream, Dim3(blocks), 64, 0, G1EncodeBody(), (const G1Affine*)pts.p, (uint32_t)count, enc.p, (uint8_t*)nullptr);
    d2h(ctx->stream, ok_out, ok.p, count);
    d2h(ctx->stream, out_be96, enc.p, count * 96);
    stream_sync(ctx->stream);
    DR_API_END
}

// ---------------------------------------------------------------------------------------- NTT
int dr_fr_ntt(dr_ctx* c, uint8_t* data_le32, size_t n, size_t batch, int inverse, const uint8_t omega_le32[32]) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || !data_le32 || !omega_le32) throw Error(DR_EINVAL, "bad argument");
    if (n < 2 || n > (1u << 22) || (n & (n - 1))) throw Error(DR_EINVAL, "n must be a power of two in [2, 2^22]");
    ctx->activate();
    if (!batch) return DR_OK;
    Fr om;
    fr_from_le_bytes_raw(om, omega_le32);
    if (!om.is_canonical_raw()) throw Error(DR_EINVAL, "omega is not canonical");
    om = om.to_mont();
    const NttPlan& plan = ctx->plan((uint32_t)n, om);
    size_t total = n * batch;
    DevBuf<uint8_t> raw(total * 32);
    DevBuf<Fr> buf(total), tmp;
    h2d(ctx->stream, raw.p, data_le32, total * 32);
    uint32_t blocks = (uint32_t)((total + 255) / 256);
    launch(ctx->stream, Dim3(blocks), 256, 0, FrToMontBody(), (const uint8_t*)raw.p, buf.p, total, (uint32_t*)nullptr);
    ntt_device(ctx, plan, buf.p, buf.p, batch, inverse != 0, tmp);
    launch(ctx->stream, Dim3(blocks), 256, 0, FrFromMontBody(), (const Fr*)buf.p, raw.p, total);
    d2h(ctx->stream, data_le32, raw.p, total * 32);
    stream_sync(ctx->stream);
    DR_API_END
}

// Device-resident timing of the batched transform (HBM / integer roofline of the NTT passes): `batch` vectors of n
// pseudo-random elements, `iters` forward transforms; returns ms per iteration and a checksum element.
int dr_fr_ntt_bench(dr_ctx* c, size_t n, size_t batch, int iters, const uint8_t omega_le32[32], float* ms_per_iter, uint8_t first_le32[32]) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || !omega_le32 || iters <= 0 || n < 2 || n > (1u << 22) || (n & (n - 1)) || !batch) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    Fr om;
    fr_from_le_bytes_raw(om, omega_le32);
    if (!om.is_canonical_raw()) throw Error(DR_EINVAL, "omega is not canonical");
    om = om.to_mont();
    const NttPlan& plan = ctx->plan((uint32_t)n, om);
    size_t total = n * batch;
    std::vector<uint8_t> host(total * 32);
    uint64_t st = 0x1234567ULL + n;
    for (size_t i = 0; i < total; i++) {
        uint64_t w[4] = {splitmix64(st), splitmix64(st), splitmix64(st), splitmix64(st) >> 2};
        memcpy(&host[32 * i], w, 32);
    }
    DevBuf<uint8_t> raw(total * 32);
    DevBuf<Fr> a(total), b(total), tmp;
    h2d(ctx->stream, raw.p, host.data(), total * 32);
    launch(ctx->stream, Dim3((uint32_t)((total + 255) / 256)), 256, 0, FrToMontBody(), (const uint8_t*)raw.p, a.p, total, (uint32_t*)nullptr);
    ntt_device(ctx, plan, a.p, b.p, batch, false, tmp);  // warm-up (also sizes tmp)
    stream_sync(ctx->stream);
    float ms = 0;
    dr_ctx_timer_start(c);
    for (int it = 0; it < iters; it++) ntt_device(ctx, plan, a.p, b.p, batch, false, tmp);
    dr_ctx_timer_stop(c, &ms);
    if (ms_per_iter) *ms_per_iter = ms / iters;
    if (first_le32) {
        launch(ctx->stream, Dim3(1), 32, 0, FrFromMontBody(), (const Fr*)b.p, raw.p, (size_t)1);
        d2h(ctx->stream, first_le32, raw.p, 32);
        stream_sync(ctx->stream);
    }
    DR_API_END
}

}  // extern "C"
