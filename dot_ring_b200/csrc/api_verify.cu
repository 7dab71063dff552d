// C ABI, part 5: verification side -- pairing checks, Pedersen / Tiny VRF batch verification, ring-proof verification.
#include "api_internal.cuh"
#include "pairing.cuh"
#include "ring.cuh"

namespace dr {

// one thread per check: equal[i] = ( e(a1_i, b1_i) == e(a2_i, b2_i) ); bad[i] = 1 on a malformed encoding
struct PairingCheckBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* a1, const uint8_t* b1, const uint8_t* a2, const uint8_t* b2, uint32_t n, PairingConsts k, uint8_t* equal,
                          uint8_t* bad) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < n) {
                G1Affine p1, p2;
                G2Affine q1, q2;
                bool ok = g1_decode(p1, a1 + 96 * (size_t)i, 96) && g1_decode(p2, a2 + 96 * (size_t)i, 96) && g2_decode_uncompressed(q1, b1 + 192 * (size_t)i) &&
                          g2_decode_uncompressed(q2, b2 + 192 * (size_t)i);
                bad[i] = ok ? 0 : 1;
                equal[i] = (ok && pairing_equal(p1, q1, p2, q2, k)) ? 1 : 0;
            }
        }
    }
};


std::shared_ptr<Ctx::G2Lines> Ctx::pairing_lines(const uint8_t* g2_be192, const G2Affine g2[2]) {
    for (auto& l : g2_lines)
        if (!memcmp(l->g2_be192, g2_be192, 384)) return l;
    auto l = std::make_shared<G2Lines>();
    memcpy(l->g2_be192, g2_be192, 384);
    std::vector<LineCoeffs> host(2 * MILLER_LINES);
    miller_precompute_lines(g2[0], host.data());
    miller_precompute_lines(g2[1], host.data() + MILLER_LINES);
    l->lines.alloc(host.size());
    h2d(stream, l->lines.p, host.data(), host.size() * sizeof(LineCoeffs));
    stream_sync(stream);
    if (g2_lines.size() >= FIXED_TABLE_CAP) g2_lines.erase(g2_lines.begin());
    g2_lines.push_back(l);
    return l;
}

VerifierKeyDev make_verifier_key(Ctx* ctx, uint32_t N, const Fr& omega, const TEAffine& seed, const uint8_t* label, uint32_t label_len, const uint8_t* g1_0_be96,
                                 const uint8_t* g2_be192, const uint8_t* fixed_be96, std::shared_ptr<Ctx::G2Lines>& lines) {
    if (N < 8 || (N & (N - 1))) throw Error(DR_EINVAL, "domain_size must be a power of two");
    VerifierKeyDev vk{};
    vk.N = N;
    vk.logN = 0;
    while ((1u << vk.logN) < N) vk.logN++;
    vk.omega = omega;
    check_primitive_root(omega, vk.logN);
    domain_tail(omega, vk.tail, vk.w_last);
    vk.n_inv = Fr::from_u32(N).inv();
    vk.seed = seed;
    for (int i = 0; i < 3; i++)
        if (!g1_decode(vk.fixed[i], fixed_be96 + 96 * i, 96)) throw Error(DR_EINVAL, "invalid BLS12-381 G1 encoding in verifier key");
    if (!g1_decode(vk.fixed[3], g1_0_be96, 96) || vk.fixed[3].is_inf()) throw Error(DR_EINVAL, "invalid BLS12-381 G1 encoding in verifier key");
    for (int i = 0; i < 2; i++)
        if (!g2_decode_uncompressed(vk.g2[i], g2_be192 + 192 * i)) throw Error(DR_EINVAL, "invalid BLS12-381 G2 encoding in verifier key");
    vk.pc = ctx->pairing_consts();
    lines = ctx->pairing_lines(g2_be192, vk.g2);  // once per context and G2 pair
    vk.lines = lines->lines.p;
    vk.prefix = ring_transcript_prefix(label, label_len, g1_0_be96, g2_be192, fixed_be96);
    return vk;
}

// cooperative verification kernels: eight lanes per item (te_coop.cuh), eight items per block.  They cut the latency of an item
// 3 - 4x but keep at most five of eight lanes busy, so batches large enough to fill the machine with one item per thread
// (measured cross-over: a few thousand items) use the serial kernels.
constexpr uint32_t VRF_VERIFY_THREADS = 64, VRF_VERIFY_ITEMS = VRF_VERIFY_THREADS / COOP_LANES;
static std::atomic<size_t> VRF_VERIFY_COOP_BELOW{8192};

static void launch_pedersen_verify(Ctx* ctx, Stream st, SuiteDev su, const VerifyInput* in, const uint8_t* blob, const uint8_t* proofs, uint32_t stride, const TEAffine* pts,
                                   const uint8_t* ok, uint32_t m, uint32_t* status) {
    auto g_table = ctx->fixed_table(su.generator), b_table = ctx->fixed_table(su.blinding_base);  // the context keeps them alive
    su.g_tab = g_table->tab.p;
    su.b_tab = b_table->tab.p;
    if (m >= VRF_VERIFY_COOP_BELOW.load()) {
        launch(st, Dim3((m + 63) / 64), 64, 0, PedersenVerifySerialBody(), su, in, blob, proofs, stride, pts, ok, m, status);
        return;
    }
    launch(st, Dim3((m + VRF_VERIFY_ITEMS - 1) / VRF_VERIFY_ITEMS), VRF_VERIFY_THREADS, vrf_verify_coop_smem(VRF_VERIFY_THREADS), PedersenVerifyBody(), su, in, blob, proofs, stride,
           pts, ok, m, status);
}

// uploads the per-item (offset, length) table and the blob; returns the device buffers
struct ItemsDev {
    DevBuf<VerifyInput> in;
    DevBuf<uint8_t> blob;
};
static void upload_items(Ctx* ctx, ItemsDev& d, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off, const uint32_t* ad_len) {
    if (!in_off || !in_len || !ad_off || !ad_len) throw Error(DR_EINVAL, "bad argument");
    std::vector<VerifyInput> h(n);
    size_t blob_len = 0;
    for (size_t i = 0; i < n; i++) {
        h[i] = {in_off[i], in_len[i], ad_off[i], ad_len[i]};
        size_t e1 = (size_t)in_off[i] + in_len[i], e2 = (size_t)ad_off[i] + ad_len[i];
        if (e1 > blob_len) blob_len = e1;
        if (e2 > blob_len) blob_len = e2;
    }
    if (blob_len && !blob) throw Error(DR_EINVAL, "null blob");
    d.in.alloc(n);
    d.blob.alloc(blob_len ? blob_len : 1);
    h2d(ctx->stream, d.in.p, h.data(), n * sizeof(VerifyInput));
    h2d(ctx->stream, d.blob.p, blob, blob_len);
    stream_sync(ctx->stream);  // h goes out of scope
}

static void status_to_verdict(const std::vector<uint32_t>& st, uint8_t* verdict) {
    for (size_t i = 0; i < st.size(); i++) verdict[i] = (st[i] & ST_MALFORMED) ? 2 : st[i] ? 0 : 1;
}

// aggregated batches of at least this many proofs fold their sides with two bucket-method MSMs (the MSM pipeline has a
// latency floor of a few ms, below this size the per-proof scalar multiplications are faster); tests lower it
static std::atomic<size_t> RING_VERIFY_MSM_THRESHOLD{8192};  // process-wide test knob; read once per call

// The verifier keys of one verification call: a device table of nkeys keys and, per item, the index of its key.
struct VerifyKeys {
    const VerifierKeyDev* table = nullptr;  // device
    uint32_t nkeys = 1;
    const uint32_t* index = nullptr;       // device, one entry per item; nullptr: every item uses table[0]
    const uint32_t* host_index = nullptr;  // the same on the host (grouping of the two-MSM route)
    const LineCoeffs* lines = nullptr;     // Miller-loop lines of the G2 points every key shares (aggregated check)
};

// shared tail of the ring-verification entry points; relations / payloads already on the device
static void ring_proof_verify_device(Ctx* ctx, const VerifyKeys& keys, size_t n, const uint8_t* payloads, uint32_t stride, const TEAffine* relations, uint32_t rel_stride,
                                     const uint8_t* coeffs_le32, const uint32_t* extra_status, int aggregate, uint8_t* verdict, int* all_ok, bool extra_on_side = false) {
    // extra_on_side: extra_status is being written by work on ctx->side (forked by the caller); joined before its first reader
    struct SideJoin {  // an exception below must not leave the side stream running into freed buffers
        Ctx* c;
        bool pending;
        ~SideJoin() {
            if (pending) c->join_side();
        }
    } side_join{ctx, extra_on_side};
    if (!coeffs_le32) throw Error(DR_EINVAL, "random batching coefficients are required (2 x 32 bytes per proof)");
    for (size_t i = 0; i < 2 * n; i++) {
        Fr r;
        fr_from_le_bytes_raw(r, coeffs_le32 + 32 * i);
        if (!r.is_canonical_raw() || r.is_zero()) throw Error(DR_EINVAL, "batching coefficients must be canonical and non-zero");
    }
    DevBuf<VerifyState> vs(n);
    DevBuf<uint8_t> dco(n * 64), dverdict(n);
    DevBuf<uint32_t> dall(1);
    dev_zero(ctx->stream, vs.p, n * sizeof(VerifyState));
    h2d(ctx->stream, dco.p, coeffs_le32, n * 64);
    const uint32_t m = (uint32_t)n;
    launch(ctx->stream, Dim3((7 * m + 63) / 64), 64, 0, PayloadG1DecodeBody(), payloads, stride, m, vs.p);
    // the subgroup tests of the decoded points overlap the transcript algebra; joined before the G1 terms read them
    struct Side2Join {
        Ctx* c;
        bool pending;
        ~Side2Join() {
            if (pending) c->join_side2();
        }
    } side2_join{ctx, true};
    ctx->fork_side2();
    launch(ctx->side2, Dim3((7 * m + 63) / 64), 64, 0, PayloadG1SubgroupBody(), m, vs.p);
    launch(ctx->stream, Dim3((m + 63) / 64), 64, 0, RingVerifyAlgebraBody(), keys.table, keys.index, payloads, stride, relations, rel_stride, (const uint8_t*)dco.p, m, vs.p);
    ctx->join_side2();
    side2_join.pending = false;
    uint32_t all = 0;
    const bool by_msm = aggregate && n >= RING_VERIFY_MSM_THRESHOLD.load();
    if (!by_msm) launch(ctx->stream, Dim3((2 * VERIFY_TERMS * m + 63) / 64), 64, 0, RingVerifyTermsBody(), keys.table, keys.index, m, vs.p);
    if (side_join.pending) {
        ctx->join_side();
        side_join.pending = false;
    }
    if (by_msm) {
        // two variable-base MSMs instead of 13 scalar multiplications per proof; the fixed commitments enter once per key, with
        // the scalars of that key's proofs summed (proofs grouped by key: grouped[start[k] .. start[k + 1]))
        const uint32_t threads = 64, nparts = (m + threads - 1) / threads, K = keys.nkeys;
        const size_t n_lhs = 7 * n + 3 * (size_t)K + 1;
        DevBuf<G1Affine> lhs_pts(n_lhs), rhs_pts(2 * n), sides(2);
        DevBuf<uint8_t> lhs_sc(32 * n_lhs), rhs_sc(32 * 2 * n);
        DevBuf<Fr> fixed_sc(3 * n), one_partial(nparts);
        DevBuf<G1> partial(2);
        DevBuf<uint32_t> bad(1), dstart, dgrouped;
        if (keys.index) {
            std::vector<uint32_t> start(K + 1, 0), grouped(n);
            for (size_t i = 0; i < n; i++) start[keys.host_index[i] + 1]++;
            for (uint32_t k = 0; k < K; k++) start[k + 1] += start[k];
            std::vector<uint32_t> fill(start.begin(), start.end() - 1);
            for (size_t i = 0; i < n; i++) grouped[fill[keys.host_index[i]]++] = (uint32_t)i;
            dstart.alloc(K + 1);
            dgrouped.alloc(n);
            h2d(ctx->stream, dstart.p, start.data(), (K + 1) * sizeof(uint32_t));
            h2d(ctx->stream, dgrouped.p, grouped.data(), n * sizeof(uint32_t));
            stream_sync(ctx->stream);  // start / grouped go out of scope
        }
        dev_zero(ctx->stream, bad.p, 4);
        launch(ctx->stream, Dim3(nparts), threads, threads * sizeof(Fr), RingVerifyGatherBody(), m, (const VerifyState*)vs.p, extra_status, dverdict.p, lhs_pts.p, lhs_sc.p,
               rhs_pts.p, rhs_sc.p, fixed_sc.p, one_partial.p, bad.p);
        launch(ctx->stream, Dim3(K), threads, 3 * threads * sizeof(Fr), RingVerifyFixedBody(), keys.table, K, (const uint32_t*)dstart.p, (const uint32_t*)dgrouped.p, m,
               (const Fr*)fixed_sc.p, (const Fr*)one_partial.p, nparts, lhs_pts.p, lhs_sc.p);
        msm_points_device(ctx, lhs_pts.p, lhs_sc.p, n_lhs, sides.p);
        msm_points_device(ctx, rhs_pts.p, rhs_sc.p, 2 * n, sides.p + 1);
        launch(ctx->stream, Dim3(1), 32, 0, RingVerifySidesFromAffineBody(), (const G1Affine*)sides.p, partial.p);
        launch(ctx->stream, Dim3(1), 32, ring_verify_warp_smem(), RingVerifyAggregateBody(), keys.lines, ctx->pairing_consts(), (const G1*)partial.p, 1u, (const uint32_t*)bad.p, dall.p);
        d2h(ctx->stream, &all, dall.p, 4);
        d2h(ctx->stream, verdict, dverdict.p, n);
        stream_sync(ctx->stream);
    } else if (aggregate) {
        const uint32_t threads = 64;
        uint32_t nparts = (m + 4 * threads - 1) / (4 * threads);
        if (nparts > 64) nparts = 64;
        DevBuf<G1> partial(2 * (size_t)nparts);
        DevBuf<uint32_t> bad(1);
        dev_zero(ctx->stream, bad.p, 4);
        launch(ctx->stream, Dim3(nparts), threads, 2 * threads * sizeof(G1), RingVerifyPartialSumBody(), m, (const VerifyState*)vs.p, extra_status, dverdict.p, partial.p, bad.p);
        launch(ctx->stream, Dim3(1), 32, ring_verify_warp_smem(), RingVerifyAggregateBody(), keys.lines, ctx->pairing_consts(), (const G1*)partial.p, nparts, (const uint32_t*)bad.p, dall.p);
        d2h(ctx->stream, &all, dall.p, 4);
        d2h(ctx->stream, verdict, dverdict.p, n);
        stream_sync(ctx->stream);  // partial / bad go out of scope
    } else {
#ifndef DR_PAIRING_MINB
#define DR_PAIRING_MINB 8
#endif
        launch_lb<32, DR_PAIRING_MINB>(ctx->stream, Dim3(m), 32, ring_verify_warp_smem(), RingVerifyFinishBody(), keys.table, keys.index, m, (const VerifyState*)vs.p,
                                       extra_status, dverdict.p);
    }
    d2h(ctx->stream, verdict, dverdict.p, n);
    stream_sync(ctx->stream);
    if (!aggregate) {
        all = 1;
        for (size_t i = 0; i < n; i++)
            if (verdict[i] != 1) all = 0;
    }
    if (all_ok) *all_ok = (int)all;
}

// RingVRF.decode + verify / batch_verify (vrf/ring/vrf.py:60-93,226-283) of n 784-byte proofs: the Pedersen part, then the ring proof
// with the relation Ybar under the item's verifier key
static void ring_vrf_verify(Ctx* ctx, const SuiteDev& suite, const VerifyKeys& keys, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len,
                            const uint32_t* ad_off, const uint32_t* ad_len, const uint8_t* proofs784, const uint8_t* coeffs_le32, int aggregate, uint8_t* verdict,
                            int* all_ok) {
    ItemsDev items;
    upload_items(ctx, items, n, blob, in_off, in_len, ad_off, ad_len);
    const uint32_t m = (uint32_t)n;
    DevBuf<uint8_t> dpr(n * 784), dok(4 * n);
    DevBuf<TEAffine> pts(4 * n);
    DevBuf<uint32_t> dst(n);
    h2d(ctx->stream, dpr.p, proofs784, n * 784);
    launch(ctx->stream, Dim3((4 * m + 63) / 64), 64, 0, TeDecodeManyBody(), (const uint8_t*)dpr.p, 784u, 4u, 4 * m, pts.p, dok.p);
    // The Pedersen equations only meet the ring proof at the verdict, so they run on the side stream next to the payload decode, the
    // transcript algebra and the G1 terms (a single verification is a chain of latency-bound kernels: this takes the longest one
    // off the critical path; large batches lose nothing).
    ctx->fork_side();
    launch_pedersen_verify(ctx, ctx->side, suite, (const VerifyInput*)items.in.p, (const uint8_t*)items.blob.p, (const uint8_t*)dpr.p, 784u, (const TEAffine*)pts.p,
                           (const uint8_t*)dok.p, m, dst.p);
    // relation = blinded public key (second Pedersen point); payload follows the 192-byte Pedersen part
    ring_proof_verify_device(ctx, keys, n, dpr.p + 192, 784, pts.p + 1, 4, coeffs_le32, dst.p, aggregate, verdict, all_ok, true);
}

// dr_ring_verifier: the verifier key of one ring, built from its 144-byte root, and the suite of its Pedersen part
struct RingVerifier {
    Ctx* ctx = nullptr;
    VerifierKeyDev vk{};
    std::shared_ptr<Ctx::G2Lines> lines;
    SuiteDev suite{};
    uint8_t g1_0_be96[96];
};

}  // namespace dr

using namespace dr;

extern "C" {

int dr_ring_verify_set_msm_threshold(size_t n) {
    RING_VERIFY_MSM_THRESHOLD = n;
    return DR_OK;
}

int dr_vrf_verify_set_coop_threshold(size_t n) {
    VRF_VERIFY_COOP_BELOW = n;
    return DR_OK;
}

int dr_pairing_check_batch(dr_ctx* c, const uint8_t* a1_be96, const uint8_t* b1_be192, const uint8_t* a2_be96, const uint8_t* b2_be192, size_t n, uint8_t* equal) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || (n && (!a1_be96 || !b1_be192 || !a2_be96 || !b2_be192 || !equal))) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (!n) return DR_OK;
    DevBuf<uint8_t> da1(n * 96), da2(n * 96), db1(n * 192), db2(n * 192), deq(n), dbad(n);
    h2d(ctx->stream, da1.p, a1_be96, n * 96);
    h2d(ctx->stream, da2.p, a2_be96, n * 96);
    h2d(ctx->stream, db1.p, b1_be192, n * 192);
    h2d(ctx->stream, db2.p, b2_be192, n * 192);
    launch(ctx->stream, Dim3((uint32_t)((n + 31) / 32)), 32, 0, PairingCheckBody(), (const uint8_t*)da1.p, (const uint8_t*)db1.p, (const uint8_t*)da2.p, (const uint8_t*)db2.p,
           (uint32_t)n, ctx->pairing_consts(), deq.p, dbad.p);
    std::vector<uint8_t> bad(n);
    d2h(ctx->stream, equal, deq.p, n);
    d2h(ctx->stream, bad.data(), dbad.p, n);
    stream_sync(ctx->stream);
    for (size_t i = 0; i < n; i++)
        if (bad[i]) throw Error(DR_EINVAL, "invalid BLS12-381 point encoding");
    DR_API_END
}

int dr_pedersen_verify_batch(dr_ctx* c, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                             const uint32_t* ad_len, const uint8_t* proofs192, uint8_t* verdict) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || (n && (!proofs192 || !verdict))) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (!n) return DR_OK;
    SuiteDev su = suite_param(suite);
    ItemsDev items;
    upload_items(ctx, items, n, blob, in_off, in_len, ad_off, ad_len);
    const uint32_t m = (uint32_t)n;
    DevBuf<uint8_t> dpr(n * 192), dok(4 * n);
    DevBuf<TEAffine> pts(4 * n);
    DevBuf<uint32_t> dst(n);
    h2d(ctx->stream, dpr.p, proofs192, n * 192);
    launch(ctx->stream, Dim3((4 * m + 63) / 64), 64, 0, TeDecodeManyBody(), (const uint8_t*)dpr.p, 192u, 4u, 4 * m, pts.p, dok.p);
    launch_pedersen_verify(ctx, ctx->stream, su, (const VerifyInput*)items.in.p, (const uint8_t*)items.blob.p, (const uint8_t*)dpr.p, 192u, (const TEAffine*)pts.p, (const uint8_t*)dok.p, m, dst.p);
    std::vector<uint32_t> st(n);
    d2h(ctx->stream, st.data(), dst.p, n * 4);
    stream_sync(ctx->stream);
    status_to_verdict(st, verdict);
    DR_API_END
}

// thin == 0: Tiny (80-byte proofs, points O | PK per item); thin != 0: Thin (96-byte proofs, points O | R | PK)
static void ietf_verify_batch(Ctx* ctx, const dr_vrf_suite* suite, uint32_t thin, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len,
                              const uint32_t* ad_off, const uint32_t* ad_len, const uint8_t* public_keys32, const uint8_t* proofs, uint8_t* verdict) {
    if (!ctx || (n && (!public_keys32 || !proofs || !verdict))) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (!n) return;
    SuiteDev su = suite_param(suite);
    ItemsDev items;
    upload_items(ctx, items, n, blob, in_off, in_len, ad_off, ad_len);
    const uint32_t m = (uint32_t)n, npts = thin ? 3 : 2, plen = thin ? 96 : 80;
    // interleave the proof's points and the public key so one decode launch covers them all
    std::vector<uint8_t> enc((size_t)32 * npts * n);
    for (size_t i = 0; i < n; i++) {
        memcpy(&enc[32 * npts * i], proofs + plen * i, 32 * (npts - 1));
        memcpy(&enc[32 * npts * i + 32 * (npts - 1)], public_keys32 + 32 * i, 32);
    }
    DevBuf<uint8_t> denc(enc.size()), dpr((size_t)plen * n), dok((size_t)npts * n);
    DevBuf<TEAffine> pts((size_t)npts * n);
    DevBuf<uint32_t> dst(n);
    h2d(ctx->stream, denc.p, enc.data(), enc.size());
    h2d(ctx->stream, dpr.p, proofs, (size_t)plen * n);
    launch(ctx->stream, Dim3((npts * m + 63) / 64), 64, 0, TeDecodeManyBody(), (const uint8_t*)denc.p, 32u * npts, npts, npts * m, pts.p, dok.p);
    auto g_table = ctx->fixed_table(su.generator);  // s * G of the large-batch kernel comes from the window table
    su.g_tab = g_table->tab.p;
    if (m >= VRF_VERIFY_COOP_BELOW.load())
        launch(ctx->stream, Dim3((m + 63) / 64), 64, 0, IetfVerifySerialBody(), su, thin, (const VerifyInput*)items.in.p, (const uint8_t*)items.blob.p, (const uint8_t*)dpr.p,
               (const TEAffine*)pts.p, (const uint8_t*)dok.p, m, dst.p);
    else
        launch(ctx->stream, Dim3((m + VRF_VERIFY_ITEMS - 1) / VRF_VERIFY_ITEMS), VRF_VERIFY_THREADS, vrf_verify_coop_smem(VRF_VERIFY_THREADS), IetfVerifyBody(), su, thin,
               (const VerifyInput*)items.in.p, (const uint8_t*)items.blob.p, (const uint8_t*)dpr.p, (const TEAffine*)pts.p, (const uint8_t*)dok.p, m, dst.p);
    std::vector<uint32_t> st(n);
    d2h(ctx->stream, st.data(), dst.p, n * 4);
    stream_sync(ctx->stream);
    status_to_verdict(st, verdict);
}

int dr_tiny_verify_batch(dr_ctx* c, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                         const uint32_t* ad_len, const uint8_t* public_keys32, const uint8_t* proofs80, uint8_t* verdict) {
    DR_API_BEGIN
    ietf_verify_batch((Ctx*)c, suite, 0, n, blob, in_off, in_len, ad_off, ad_len, public_keys32, proofs80, verdict);
    DR_API_END
}

int dr_thin_verify_batch(dr_ctx* c, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                         const uint32_t* ad_len, const uint8_t* public_keys32, const uint8_t* proofs96, uint8_t* verdict) {
    DR_API_BEGIN
    ietf_verify_batch((Ctx*)c, suite, 1, n, blob, in_off, in_len, ad_off, ad_len, public_keys32, proofs96, verdict);
    DR_API_END
}

// kind 0: Pedersen (192-byte proofs), 1: Tiny (80-byte proofs), 2: Thin (96-byte proofs)
static void vrf_prove_batch(Ctx* ctx, const dr_vrf_suite* suite, int kind, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len,
                            const uint32_t* ad_off, const uint32_t* ad_len, const uint8_t* sks32, uint8_t* out, uint8_t* blinding32 = nullptr) {
    if (!ctx || (n && (!sks32 || !out))) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (!n) return;
    SuiteDev su = suite_param(suite);
    auto g_table = ctx->fixed_table(su.generator), b_table = ctx->fixed_table(su.blinding_base);
    su.g_tab = g_table->tab.p;
    su.b_tab = b_table->tab.p;
    ItemsDev items;
    upload_items(ctx, items, n, blob, in_off, in_len, ad_off, ad_len);
    const size_t len = kind == 0 ? 192 : kind == 1 ? 80 : 96;
    DevBuf<uint8_t> dsk(n * 32), dout(n * len), dbl(blinding32 ? n * 32 : 1);
    h2d(ctx->stream, dsk.p, sks32, n * 32);
    const uint32_t m = (uint32_t)n;
    if (kind == 0)
        launch(ctx->stream, Dim3((m + 63) / 64), 64, 0, PedersenProveStandaloneBody(), su, (const VerifyInput*)items.in.p, (const uint8_t*)items.blob.p, (const uint8_t*)dsk.p, m, dout.p,
               blinding32 ? dbl.p : (uint8_t*)nullptr);
    else
        launch(ctx->stream, Dim3((m + 63) / 64), 64, 0, IetfProveBody(), su, kind == 2 ? 1u : 0u, (const VerifyInput*)items.in.p, (const uint8_t*)items.blob.p,
               (const uint8_t*)dsk.p, m, dout.p);
    d2h(ctx->stream, out, dout.p, n * len);
    if (blinding32) d2h(ctx->stream, blinding32, dbl.p, n * 32);
    dev_zero(ctx->stream, dsk.p, n * 32);  // the cached block must not hand secret keys to a later call
    if (blinding32) dev_zero(ctx->stream, dbl.p, n * 32);
    stream_sync(ctx->stream);
}

int dr_pedersen_prove_batch_ex(dr_ctx* c, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                               const uint32_t* ad_len, const uint8_t* secret_keys32, uint8_t* proofs192, uint8_t* blinding32) {
    DR_API_BEGIN
    vrf_prove_batch((Ctx*)c, suite, 0, n, blob, in_off, in_len, ad_off, ad_len, secret_keys32, proofs192, blinding32);
    DR_API_END
}

int dr_pedersen_prove_batch(dr_ctx* c, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                            const uint32_t* ad_len, const uint8_t* secret_keys32, uint8_t* proofs192) {
    DR_API_BEGIN
    vrf_prove_batch((Ctx*)c, suite, 0, n, blob, in_off, in_len, ad_off, ad_len, secret_keys32, proofs192);
    DR_API_END
}

int dr_tiny_prove_batch(dr_ctx* c, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                        const uint32_t* ad_len, const uint8_t* secret_keys32, uint8_t* proofs80) {
    DR_API_BEGIN
    vrf_prove_batch((Ctx*)c, suite, 1, n, blob, in_off, in_len, ad_off, ad_len, secret_keys32, proofs80);
    DR_API_END
}

int dr_thin_prove_batch(dr_ctx* c, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                        const uint32_t* ad_len, const uint8_t* secret_keys32, uint8_t* proofs96) {
    DR_API_BEGIN
    vrf_prove_batch((Ctx*)c, suite, 2, n, blob, in_off, in_len, ad_off, ad_len, secret_keys32, proofs96);
    DR_API_END
}

int dr_ring_proof_verify_batch(dr_ctx* c, const dr_verifier_key* key, size_t n, const uint8_t* relations_xy64, const uint8_t* payloads592, const uint8_t* coeffs_le32,
                               int aggregate, uint8_t* verdict, int* all_ok) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || !key || (n && (!relations_xy64 || !payloads592 || !verdict))) throw Error(DR_EINVAL, "bad argument");
    if (key->label_len > 32) throw Error(DR_EINVAL, "transcript label too long");
    ctx->activate();
    if (all_ok) *all_ok = 1;
    if (!n) return DR_OK;
    std::shared_ptr<Ctx::G2Lines> lines;
    VerifierKeyDev vk = make_verifier_key(ctx, key->domain_size, fr_param(key->omega), te_param(key->seed), key->label, key->label_len, key->g1_0_be96, key->g2_be192,
                                          key->fixed_be96, lines);
    DevBuf<VerifierKeyDev> dvk(1);
    h2d(ctx->stream, dvk.p, &vk, sizeof(VerifierKeyDev));
    VerifyKeys keys;
    keys.table = dvk.p;
    keys.lines = vk.lines;
    std::vector<TEAffine> rel(n);
    for (size_t i = 0; i < n; i++) rel[i] = {fr_param(relations_xy64 + 64 * i), fr_param(relations_xy64 + 64 * i + 32)};
    DevBuf<TEAffine> drel(n);
    DevBuf<uint8_t> dpl(n * 592);
    h2d(ctx->stream, drel.p, rel.data(), n * sizeof(TEAffine));
    h2d(ctx->stream, dpl.p, payloads592, n * 592);
    ring_proof_verify_device(ctx, keys, n, dpl.p, 592, drel.p, 1, coeffs_le32, nullptr, aggregate, verdict, all_ok);
    DR_API_END
}

int dr_ring_verify_batch(dr_ctx* c, dr_ring* r, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off, const uint32_t* ad_len,
                         const uint8_t* proofs784, const uint8_t* coeffs_le32, int aggregate, uint8_t* verdict, int* all_ok) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    Ring* ring = (Ring*)r;
    if (!ctx || !ring || (n && (!proofs784 || !verdict))) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (all_ok) *all_ok = 1;
    if (!n) return DR_OK;
    VerifyKeys keys;
    keys.table = ring->vk_dev.p;
    keys.lines = ring->vk.lines;
    ring_vrf_verify(ctx, ring->suite, keys, n, blob, in_off, in_len, ad_off, ad_len, proofs784, coeffs_le32, aggregate, verdict, all_ok);
    DR_API_END
}

int dr_ring_verifier_create(dr_ctx* c, const dr_ring_params* prm, const uint8_t* g1_0_be96, const uint8_t* g2_be192, const uint8_t root144[144], dr_ring_verifier** out) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || !prm || !g1_0_be96 || !g2_be192 || !root144 || !out) throw Error(DR_EINVAL, "bad argument");
    check_domain_size(prm->domain_size);
    ctx->activate();
    auto v = std::make_unique<RingVerifier>();
    v->ctx = ctx;
    v->suite = suite_param(*prm);
    // RingRoot.decode (root.py:89-109): three compressed points, no subgroup check (blst); the transcript absorbs their
    // uncompressed encodings
    uint8_t fixed_be96[288];
    for (int i = 0; i < 3; i++) {
        G1Affine a;
        if (!g1_decode(a, root144 + 48 * i, 48)) throw Error(DR_EINVAL, "invalid BLS12-381 G1 encoding in ring root");
        g1_serialize(fixed_be96 + 96 * i, a);
    }
    v->vk = make_verifier_key(ctx, prm->domain_size, fr_param(prm->omega), te_param(prm->seed), prm->suite_id, prm->suite_id_len, g1_0_be96, g2_be192, fixed_be96, v->lines);
    for (int i = 0; i < 3; i++) v->vk.fixed_outside[i] = g1_in_subgroup(v->vk.fixed[i]) ? 0 : 1;
    memcpy(v->g1_0_be96, g1_0_be96, 96);
    *out = (dr_ring_verifier*)v.release();
    DR_API_END
}

void dr_ring_verifier_destroy(dr_ring_verifier* v) { delete (RingVerifier*)v; }

int dr_ring_verify_multi(dr_ctx* c, dr_ring_verifier* const* verifiers, size_t n_verifiers, const uint32_t* verifier_index, size_t n, const uint8_t* blob,
                         const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off, const uint32_t* ad_len, const uint8_t* proofs784, const uint8_t* coeffs_le32,
                         int aggregate, uint8_t* verdict, int* all_ok) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || !verifiers || !n_verifiers || n_verifiers > UINT32_MAX || (n && (!verifier_index || !proofs784 || !verdict))) throw Error(DR_EINVAL, "bad argument");
    const RingVerifier* first = (const RingVerifier*)verifiers[0];
    for (size_t k = 0; k < n_verifiers; k++) {
        const RingVerifier* v = (const RingVerifier*)verifiers[k];
        if (!v) throw Error(DR_EINVAL, "bad argument");
        if (v->ctx != ctx) throw Error(DR_EINVAL, "ring verifier belongs to another context");
        if (!same_suite(v->suite, first->suite)) throw Error(DR_EINVAL, "ring verifiers of one call must share the suite");
        if (memcmp(v->g1_0_be96, first->g1_0_be96, 96) || memcmp(v->lines->g2_be192, first->lines->g2_be192, 384))
            throw Error(DR_EINVAL, "ring verifiers of one call must share [1]_1 and the G2 points");
    }
    for (size_t i = 0; i < n; i++)
        if (verifier_index[i] >= n_verifiers) throw Error(DR_EINVAL, "verifier index out of range");
    ctx->activate();
    if (all_ok) *all_ok = 1;
    if (!n) return DR_OK;
    std::vector<VerifierKeyDev> table(n_verifiers);
    for (size_t k = 0; k < n_verifiers; k++) table[k] = ((const RingVerifier*)verifiers[k])->vk;
    DevBuf<VerifierKeyDev> dtable(n_verifiers);
    DevBuf<uint32_t> dindex(n);
    h2d(ctx->stream, dtable.p, table.data(), n_verifiers * sizeof(VerifierKeyDev));
    h2d(ctx->stream, dindex.p, verifier_index, n * sizeof(uint32_t));
    VerifyKeys keys;
    keys.table = dtable.p;
    keys.nkeys = (uint32_t)n_verifiers;
    keys.index = dindex.p;
    keys.host_index = verifier_index;
    keys.lines = first->vk.lines;
    ring_vrf_verify(ctx, first->suite, keys, n, blob, in_off, in_len, ad_off, ad_len, proofs784, coeffs_le32, aggregate, verdict, all_ok);
    DR_API_END
}

}  // extern "C"
