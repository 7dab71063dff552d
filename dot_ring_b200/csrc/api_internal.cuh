// Internal host-side state shared by the api_*.cu translation units.
#pragma once
#include <chrono>
#include <memory>
#include <mutex>
#include <set>
#include <string>
#include <vector>

#include "../../include/dot_ring_b200.h"
#include "fp.cuh"
#include "g1.cuh"
#include "hash.cuh"
#include "msm.cuh"
#include "ntt.cuh"
#include "pairing.cuh"
#include "ring.cuh"
#include "rt.cuh"
#include "te.cuh"
#include "verify.cuh"

namespace dr {

#ifndef DR_COMMIT_THREADS
#define DR_COMMIT_THREADS 128  // A/B builds: NVCC_EXTRA="-DDR_COMMIT_THREADS=96 -DDR_COMMIT_MINB=5"
#endif
constexpr uint32_t COMMIT_THREADS = DR_COMMIT_THREADS;

int set_error(int code, const std::string& msg);

struct NttPlan {
    uint32_t n = 0, logn = 0;
    Fr omega;
    DevBuf<Fr> tw_fwd, tw_inv, n_inv;  // n <= 4096: [w^k], [w^-k] for k < n/2
    // n > 4096 (two-pass transform, ntt.cuh): n = n1 * n2; index 0 forward, 1 inverse
    uint32_t n1 = 0, n2 = 0, logn1 = 0, logn2 = 0;
    DevBuf<Fr> wfull[2], tw1[2], tw2[2];
};


struct Ctx;

// Accumulates device time per pipeline phase with events recorded between the launches.
struct PhaseTimer {
    // 0..5: pipeline phases (dr_ring_prove_phase_ms); 6: the dense commit kernel alone (CommitBodyT launches); 7: call entry -> first
    // phase of a pass (input copies, set-up); 8: last phase -> results on the host (output copies, side stream join, final sync)
    static constexpr int NPH = 9;
    float total[NPH] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t kernel_launches = 0;  // CommitBodyT launches counted into total[6]
    bool active = false;           // between reset() and the last collect() of a prove call
    int current = -1;
    std::vector<int> phase_of;  // phase that starts at mark i (-1 = end marker)
#if !defined(DR_HOST_EMULATION)
    std::vector<cudaEvent_t> events;
#else
    std::vector<std::chrono::steady_clock::time_point> stamps;
#endif
    void reset() {
        for (float& t : total) t = 0;
        phase_of.clear();
        kernel_launches = 0;
        current = -1;
    }
    void mark(Ctx* ctx, int phase);
    void collect(Ctx* ctx);
    int current_of(size_t i) const;
};

struct Ctx {
    int device = 0;
    Stream stream{};
    // work that nothing on the main stream waits for until the end of a pass (second half of the Pedersen prover) runs here
    Stream side{};
    // a second one for work that overlaps a shorter stretch of the main stream (witness interpolation next to the witness commitments)
    Stream side2{};
#if !defined(DR_HOST_EMULATION)
    cudaEvent_t ev_fork{}, ev_join{}, ev_fork2{}, ev_join2{};
    cudaEvent_t ev_start{}, ev_stop{};
#else
    std::chrono::steady_clock::time_point t_start;
#endif
    std::vector<std::unique_ptr<NttPlan>> plans;
    DevBuf<G1> partials;
    PhaseTimer phases;
    std::shared_ptr<void> prove_scratch;
    size_t prove_chunk = 0;
    int commit_mode = 0;  // 0: XYZZ accumulation (CommitBody), 1: batched-affine pairing rounds (CommitAffineBody)
    DevBuf<uint32_t> aff_refs;
    DevBuf<Fq> aff_prefix;
    DevBuf<G1Affine> aff_a, aff_b;
    bool dense_witness_commit = false;
    bool generic_ntt_path = false;  // force the large-domain route (element-wise twists + ntt_device) at any N: tests  // A/B + cross-check: commit witness columns from coefficients like the reference
    // te_mul_fixed window tables, one per distinct base point seen by this context (generators and blinding bases of the
    // suites in use); rings and running calls share ownership, the context keeps the most recent FIXED_TABLE_CAP
    struct FixedTable {
        TEAffine base;
        DevBuf<TEPre> tab;
    };
    static constexpr size_t FIXED_TABLE_CAP = 16;
    std::vector<std::shared_ptr<FixedTable>> fixed_tables;
    std::shared_ptr<FixedTable> fixed_table(const TEAffine& base);
    // Miller-loop lines of one ([1]_2, [tau]_2) pair (pairing_warp.cuh), shared by every verifier key over those points: a batch
    // that mixes rings of one SRS folds into one pairing check with one set of lines
    struct G2Lines {
        uint8_t g2_be192[384];
        DevBuf<LineCoeffs> lines;
    };
    std::vector<std::shared_ptr<G2Lines>> g2_lines;  // the most recent FIXED_TABLE_CAP pairs
    std::shared_ptr<G2Lines> pairing_lines(const uint8_t* g2_be192, const G2Affine g2[2]);
    bool have_pairing_consts = false;
    PairingConsts pairing_k;
    const PairingConsts& pairing_consts() {
        if (!have_pairing_consts) {
            pairing_k = pairing_consts_host();
            have_pairing_consts = true;
        }
        return pairing_k;
    }

    void activate() {
#if !defined(DR_HOST_EMULATION)
        DR_CUDA(cudaSetDevice(device));
        current_stream() = stream;  // the block cache orders reuse by the stream a block was freed on (rt.cuh)
#endif
    }
    uint32_t sm_count_cached = 0;
    uint32_t sm_count() {
        if (!sm_count_cached) {
            sm_count_cached = 148;
#if !defined(DR_HOST_EMULATION)
            int v = 0;
            if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && v > 0) sm_count_cached = (uint32_t)v;
#endif
        }
        return sm_count_cached;
    }
    // side stream: starts after everything queued on the main stream so far / main stream waits for everything queued on it
    void fork_side() {
#if !defined(DR_HOST_EMULATION)
        DR_CUDA(cudaEventRecord(ev_fork, stream));
        DR_CUDA(cudaStreamWaitEvent(side, ev_fork, 0));
#endif
    }
    void join_side() {
#if !defined(DR_HOST_EMULATION)
        DR_CUDA(cudaEventRecord(ev_join, side));
        DR_CUDA(cudaStreamWaitEvent(stream, ev_join, 0));
#endif
    }
    void fork_side2() {
#if !defined(DR_HOST_EMULATION)
        DR_CUDA(cudaEventRecord(ev_fork2, stream));
        DR_CUDA(cudaStreamWaitEvent(side2, ev_fork2, 0));
#endif
    }
    void join_side2() {
#if !defined(DR_HOST_EMULATION)
        DR_CUDA(cudaEventRecord(ev_join2, side2));
        DR_CUDA(cudaStreamWaitEvent(stream, ev_join2, 0));
#endif
    }
    // ms between the last fork and the completion of the side stream's work (after a stream sync); diagnostics only
    float side_span_ms() {
        float ms = 0;
#if !defined(DR_HOST_EMULATION)
        if (cudaEventElapsedTime(&ms, ev_fork, ev_join) != cudaSuccess) {
            cudaGetLastError();
            ms = -1;
        }
#endif
        return ms;
    }
    const NttPlan& plan(uint32_t n, const Fr& omega_mont);
    void release_scratch() {
        partials.release();
        aff_refs.release();
        aff_prefix.release();
        aff_a.release();
        aff_b.release();
        prove_scratch.reset();
    }
};

// Contexts created and not yet destroyed.  A ring or SRS can outlive its context (the Python wrappers are garbage-collected in any
// order), so its destroy must not touch a context that is gone.
inline std::mutex& live_ctx_mutex() {
    static std::mutex m;
    return m;
}
inline std::set<const Ctx*>& live_ctxs() {
    static std::set<const Ctx*> s;
    return s;
}
// Before an object's device buffers are freed: the block cache records a freed block on the calling thread's current stream
// (rt.cuh dev_free), and that stream may belong to a context destroyed since, possibly by another thread (an EnginePool worker
// tears its contexts down).  Free on the owning context's stream while that context is alive, else on the legacy stream.
inline void free_on_owner_stream(const Ctx* ctx) {
#if !defined(DR_HOST_EMULATION)
    std::lock_guard<std::mutex> lock(live_ctx_mutex());
    current_stream() = nullptr;
    if (ctx && live_ctxs().count(ctx)) {
        if (cudaSetDevice(ctx->device) == cudaSuccess)
            current_stream() = ctx->stream;
        else
            cudaGetLastError();  // the failure must not surface at the next launch check
    }
#else
    (void)ctx;
#endif
}

// batch transforms of `n` Montgomery elements each, in place (or in -> out); n a power of two up to 2^22
void ntt_device(Ctx* ctx, const NttPlan& plan, const Fr* in, Fr* out, size_t batch, bool inverse, DevBuf<Fr>& tmp);

// Window table of S_j = sum_{i<j} [L_i(tau)]_1, j = 1..N, for one evaluation domain (sparse witness commitments).
struct LagrangeTable {
    uint32_t N = 0;
    Fr omega;
    TableGeom geom{};
    DevBuf<G1Affine> table;
};

struct Srs {
    Ctx* ctx = nullptr;
    uint32_t n = 0;
    DevBuf<G1Affine> points;  // Montgomery affine
    DevBuf<G1Affine> table;   // fixed-base window table
    TableGeom geom{};
    uint8_t g1_0_be96[96];
    uint8_t g2_be192[384];
    std::vector<std::unique_ptr<LagrangeTable>> lagrange;
    DevBuf<LineCoeffs> lines;  // Miller-loop lines of the two G2 points (pairing_warp.cuh), built on first use
    const LineCoeffs* pairing_lines();
    // built on first use for (N, omega); tw_inv_half = [omega^-k], k < N/2, on the device
    const LagrangeTable& lagrange_table(uint32_t N, uint32_t logN, const Fr& omega, const Fr* tw_inv_half, const Fr& n_inv);
};

struct Ring {
    Ctx* ctx = nullptr;
    Srs* srs = nullptr;
    RingDev dev{};
    Fr radix_omega;  // w4 (Montgomery): rings proved in one pass must share it with omega
    DevBuf<TEAffine> nm;
    DevBuf<Fr> fixed_coef, fixed_lde, w4, w4inv;
    DevBuf<Shake128> prefix;
    RingTab tab{};            // this ring's entry of a prove call's ring table
    DevBuf<RingTab> tab_dev;  // the one-entry table of dr_ring_prove_batch
    G1Affine commitments[3];
    uint8_t commit_be96[288];
    uint8_t root144[144];
    TEAffine padding;
    const struct LagrangeTable* lag = nullptr;  // owned by the Srs (shared by every ring on the same domain)
    VerifierKeyDev vk{};
    std::shared_ptr<Ctx::G2Lines> vk_lines;
    DevBuf<VerifierKeyDev> vk_dev;  // vk on the device: the one-entry key table of the verification kernels
    SuiteDev suite{};
    std::shared_ptr<Ctx::FixedTable> g_table, b_table;
};

// Suite identity of the Pedersen part: suite id, hash-to-curve DST, hash, generator and blinding base.
inline bool same_suite(const SuiteDev& a, const SuiteDev& b) {
    return a.suite_id_len == b.suite_id_len && !memcmp(a.suite_id, b.suite_id, a.suite_id_len) && a.dst_len == b.dst_len && !memcmp(a.dst, b.dst, a.dst_len) &&
           a.hash_kind == b.hash_kind && a.generator == b.generator && a.blinding_base == b.blinding_base;
}

// ---- decoding of the parameter structs (dr_ring_params, dr_vrf_suite, dr_verifier_key) ----
inline Fr fr_param(const uint8_t* b) {
    Fr r;
    fr_from_le_bytes_raw(r, b);
    if (!r.is_canonical_raw()) throw Error(DR_EINVAL, "field element is not canonical");
    return r.to_mont();
}
inline TEAffine te_param(const uint8_t* xy) {
    TEAffine p{fr_param(xy), fr_param(xy + 32)};
    if (!te_on_curve(p)) throw Error(DR_EINVAL, "point is not on the curve");
    return p;
}
// The suite as dr_ring_params and dr_vrf_suite both carry it; the window tables are left to the caller.
inline SuiteDev suite_param(uint32_t suite_id_len, const uint8_t* suite_id, uint32_t dst_len, const uint8_t* dst, uint32_t hash_id, const uint8_t* generator,
                            const uint8_t* blinding_base) {
    if (suite_id_len > 32 || dst_len > 64) throw Error(DR_EINVAL, "suite id / DST too long");
    if (hash_id > 1) throw Error(DR_EINVAL, "unknown suite hash");
    SuiteDev d{};
    d.generator = te_param(generator);
    d.blinding_base = te_param(blinding_base);
    d.suite_id_len = suite_id_len;
    memcpy(d.suite_id, suite_id, 32);
    d.dst_len = dst_len;
    memcpy(d.dst, dst, 64);
    d.hash_kind = hash_id;
    return d;
}
inline SuiteDev suite_param(const dr_ring_params& p) {
    return suite_param(p.suite_id_len, p.suite_id, p.h2c_dst_len, p.h2c_dst, p.hash_id, p.generator, p.blinding_base);
}
inline SuiteDev suite_param(const dr_vrf_suite* s) {
    if (!s) throw Error(DR_EINVAL, "bad suite");
    return suite_param(s->suite_id_len, s->suite_id, s->h2c_dst_len, s->h2c_dst, s->hash_id, s->generator, s->blinding_base);
}
// The domain sizes a ring supports: the reference stops at 4096 (params.py:172-173); larger domains (to 2^16) run the same pipeline
// over the two-pass NTT.
inline void check_domain_size(uint32_t N) {
    if (N < 512 || N > 65536 || (N & (N - 1))) throw Error(DR_EINVAL, "domain_size must be a power of two in [512, 65536]");
}
// omega^N == 1, omega^(N/2) != 1
inline void check_primitive_root(const Fr& omega, uint32_t logN) {
    Fr t = omega;
    for (uint32_t i = 0; i + 1 < logN; i++) t = t.sqr();
    if (t == Fr::one() || t.sqr() != Fr::one()) throw Error(DR_EINVAL, "omega is not a primitive N-th root of unity");
}
// w^(N-4) and the coefficients of (X - w^(N-1))(X - w^(N-2))(X - w^(N-3)), from w^-1 (omega^N == 1)
inline void domain_tail(const Fr& omega, Fr tail[4], Fr& w_last) {
    const Fr winv = omega.inv();
    const Fr r1 = winv, r2 = winv * winv, r3 = r2 * winv;
    w_last = r3 * winv;
    tail[3] = Fr::one();
    tail[2] = (r1 + r2 + r3).neg();
    tail[1] = r1 * r2 + r1 * r3 + r2 * r3;
    tail[0] = (r1 * r2 * r3).neg();
}
// The ring transcript after the verifier key under `label` (root.py:54-71, phases.py:72-74): label | "vk" | G1[0] | G2[0..1] | the
// three fixed commitments, uncompressed.
inline Shake128 ring_transcript_prefix(const uint8_t* label, uint32_t label_len, const uint8_t* g1_0_be96, const uint8_t* g2_be192, const uint8_t* fixed_be96) {
    Shake128 tr;
    tr.init();
    tr.absorb(label, label_len);
    tr.absorb_be32(label_len);
    shake_absorb_label(tr, "vk", 2);
    tr.absorb(g1_0_be96, 96);
    tr.absorb(g2_be192, 384);
    tr.absorb(fixed_be96, 288);
    tr.absorb_be32(96 + 384 + 288);
    return tr;
}


VerifierKeyDev make_verifier_key(Ctx* ctx, uint32_t N, const Fr& omega, const TEAffine& seed, const uint8_t* label, uint32_t label_len, const uint8_t* g1_0_be96,
                                 const uint8_t* g2_be192, const uint8_t* fixed_be96, std::shared_ptr<Ctx::G2Lines>& lines);

// Fixed-base window table (msm.cuh) for n affine points already on the device.
void build_window_table(Ctx* ctx, const G1Affine* points, const TableGeom& geom, DevBuf<G1Affine>& table);

// Variable-base MSM (pippenger.cuh) over operands resident on the device: *out = sum_i scalars[i] * points[i].
void msm_points_device(Ctx* ctx, const G1Affine* points, const uint8_t* scalars_le32, size_t n, G1Affine* out);

// scalars: `batch` vectors of n Montgomery Fr, vector b at scalars + b*stride.  Result: affine points.
void commit_device(Ctx* ctx, Srs* srs, const Fr* scalars, size_t stride, uint32_t n, uint32_t batch, G1Affine* out_affine);
// two commitments of one batch with a shared finish: out_affine[0 .. batch) = first, [batch .. 2 batch) = second
void commit_device_pair(Ctx* ctx, Srs* srs, const Fr* scalars_a, size_t stride_a, uint32_t n_a, const Fr* scalars_b, size_t stride_b, uint32_t n_b, uint32_t batch,
                        G1Affine* out_affine);

}  // namespace dr

// Body of a C ABI entry point: an exception becomes its error code (DR_ECUDA for anything but dr::Error) and dr_last_error's text.
#define DR_API_BEGIN try {
#define DR_API_END                                \
    }                                             \
    catch (const dr::Error& e) {                  \
        return dr::set_error(e.code, e.what());   \
    }                                             \
    catch (const std::exception& e) {             \
        return dr::set_error(DR_ECUDA, e.what()); \
    }                                             \
    return DR_OK;
