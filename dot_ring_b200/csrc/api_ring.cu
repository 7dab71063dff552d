// C ABI, part 3: ring set-up (key ingestion, fixed columns, ring root) and batched Ring VRF proving.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "api_internal.cuh"
#include "ring.cuh"

namespace dr {

// The ring's row layout: N, padding rows, and room for the 253 bit rows next to max_ring_size keys.
static void check_ring_shape(const dr_ring_params* prm) {
    check_domain_size(prm->domain_size);
    if (prm->padding_rows != 4) throw Error(DR_EINVAL, "padding_rows must be 4 to match the 3 hidden rows");
    if (prm->max_ring_size + SCALAR_BITS + 4 > prm->domain_size) throw Error(DR_EINVAL, "max_ring_size exceeds supported size for this domain");
}

// The rows of the public vector PK || padding || 2^i B || zeros (members.py:36-53) that no key sets: padding below max_ring (a key
// overwrites its row), then the blinding-base doublings, then four zero rows.
static std::vector<TEAffine> public_vector_rows(uint32_t N, uint32_t max_ring, const TEAffine& padding, const TEAffine& blinding_base) {
    std::vector<TEAffine> host(N);
    for (uint32_t i = 0; i < max_ring; i++) host[i] = padding;
    TEExt cur = TEExt::from_affine(blinding_base);
    for (uint32_t i = max_ring; i < N - 4; i++) {
        host[i] = te_to_affine(cur);
        cur = te_dbl(cur);
    }
    for (uint32_t i = N - 4; i < N; i++) host[i] = TEAffine{Fr::zero(), Fr::zero()};
    return host;
}

// Per-pass device scratch.  Buffers with disjoint lifetimes share storage: the 16N-element low-degree extensions are dead once
// the constraints are evaluated, so the combined quotient coefficients (cagg), the aggregated opening polynomial (aggopen) and
// the linearisation polynomial (lin), all born later, live inside that block: 27 N + 1 field elements per proof instead of 35 N.
struct ProveScratch {
    size_t cap = 0;
    uint32_t N = 0;
    DevBuf<ProofState> st;
    DevBuf<ProveInput> in;
    DevBuf<Fr> wit_coef, lde, agg, quot, ntt_tmp;
    struct View {
        Fr* p = nullptr;
    } cagg, aggopen, lin;
    DevBuf<G1Affine> res;
    DevBuf<uint8_t> out, zraw, blob;
    DevBuf<uint32_t> status;
    static size_t elements_per_proof(uint32_t N) { return (size_t)27 * N + 1; }
    // A scratch sized for a larger domain fits a smaller one: every buffer holds per-proof rows of a size that grows with N, and
    // the views inside `lde` stay disjoint for any pass of at most `cap` proofs at a domain of at most N.
    bool fits(size_t n, uint32_t N_) const { return n <= cap && N_ <= N; }
    void ensure(size_t n, uint32_t N_) {
        if (fits(n, N_)) return;
        cap = n;
        N = N_;
        size_t q = 3 * (size_t)N + 1;
        st.alloc(n);
        in.alloc(n);
        wit_coef.alloc(n * 4 * N);
        lde.alloc(n * 16 * N);
        cagg.p = lde.p;                               // n x 4N
        aggopen.p = lde.p + n * 4 * (size_t)N;        // n x (3N + 1)
        lin.p = lde.p + n * (7 * (size_t)N + 1);      // n x N
        agg.alloc(n * 4 * N);
        quot.alloc(n * q);
        res.alloc(n * 4);
        out.alloc(n * 784);
        zraw.alloc(n * 12 * 32);
        status.alloc(n);
    }
};

static ProveScratch& scratch_for(Ctx* ctx) {
    if (!ctx->prove_scratch) ctx->prove_scratch = std::shared_ptr<void>(new ProveScratch(), [](void* p) { delete (ProveScratch*)p; });
    return *(ProveScratch*)ctx->prove_scratch.get();
}

// What a prove call produces.  Ring VRF (dr_ring_prove_batch / _multi): `secrets32` are secret keys, each item gets its Pedersen part
// and a 784-byte proof with a status word.  Bare ring proof (dr_ring_proof_prove_multi): `secrets32` are blinding factors, the inputs
// (blob and offsets) are unused, and each item gets its relation (64 bytes) and 592-byte payload.
struct ProveOutputs {
    bool bare = false;
    uint8_t* proofs784 = nullptr;
    uint32_t* status = nullptr;
    uint8_t* relations_xy64 = nullptr;
    uint8_t* payloads592 = nullptr;
};

// One prove call: item i against rings[ring_index[i]] (ring_index null: every item against rings[0]).  The callers have checked
// that the rings share the context, the SRS and the suite; `dtab` holds their RingTab entries on the device, in the same order.
// Items are grouped by domain size (ascending), in the caller's order within a group, and every group runs its own equal-width
// passes over one scratch sized for the largest domain of the call.  Outputs land at the caller's positions.
static void ring_prove(Ctx* ctx, Ring* const* rings, const RingTab* dtab, const uint32_t* ring_index, size_t n, const uint8_t* blob, const uint32_t* alpha_off,
                       const uint32_t* alpha_len, const uint32_t* ad_off, const uint32_t* ad_len, const uint8_t* secrets32, const uint32_t* producer_index,
                       const uint8_t* zk_rows, const ProveOutputs& res) {
    auto ring_of = [&](size_t i) { return ring_index ? ring_index[i] : 0u; };
    const bool bare = res.bare;
    const SuiteDev& suite = rings[0]->suite;
    size_t blob_len = 0;
    std::vector<uint32_t> domains;  // distinct domain sizes of the items' rings
    for (size_t i = 0; i < n; i++) {
        if (!bare) {
            size_t e1 = (size_t)alpha_off[i] + alpha_len[i], e2 = (size_t)ad_off[i] + ad_len[i];
            if (e1 > blob_len) blob_len = e1;
            if (e2 > blob_len) blob_len = e2;
        }
        const uint32_t N = rings[ring_of(i)]->dev.N;
        if (std::find(domains.begin(), domains.end(), N) == domains.end()) domains.push_back(N);
    }
    if (blob_len && !blob) throw Error(DR_EINVAL, "null blob");
    std::sort(domains.begin(), domains.end());
    // one group: the items in the caller's order, copied in and out in place; several: gathered per group and scattered back
    const bool direct = domains.size() == 1;
    std::vector<uint32_t> order;
    std::vector<size_t> group_end;
    size_t widest = n;
    if (!direct) {
        order.reserve(n);
        widest = 0;
        for (uint32_t N : domains) {
            const size_t begin = order.size();
            for (size_t i = 0; i < n; i++)
                if (rings[ring_of(i)]->dev.N == N) order.push_back((uint32_t)i);
            group_end.push_back(order.size());
            if (order.size() - begin > widest) widest = order.size() - begin;
        }
    } else {
        group_end.push_back(n);
    }
    const uint32_t N_max = domains.back();
    // (the input blob goes into a buffer that lives with the scratch: no allocation on the steady-state path)

    // proofs per pass: the one-thread-per-proof kernels (Pedersen part, witness chain, transcripts) are latency-bound, so
    // a pass should be as wide as the scratch (35 N field elements + state per proof) allows
    size_t chunk_cap = ctx->prove_chunk ? ctx->prove_chunk : 8192;
#if !defined(DR_HOST_EMULATION)
    // The free-memory query (like any allocation) can stall for tens of ms inside the driver, so it is only made when the scratch
    // has to grow: a call that fits the scratch of an earlier one reuses its pass width.
    {
        ProveScratch& cur = scratch_for(ctx);
        const size_t want = widest < chunk_cap ? widest : chunk_cap;
        if (!ctx->prove_chunk && !cur.fits(want, N_max)) {
            size_t free_b = 0, total_b = 0;
            DR_CUDA(cudaMemGetInfo(&free_b, &total_b));
            free_b += dev_cache().cached;  // recycled blocks are available to this call
            size_t per_proof = (ProveScratch::elements_per_proof(N_max) + (N_max > 4096 ? 16 * (size_t)N_max : 0)) * sizeof(Fr) + sizeof(ProofState) + 4096;
            size_t have = free_b + (cur.N == N_max ? cur.cap * per_proof : 0);
            // keep 1 GB (or half of what is left, if less) for the other buffers of this and later calls
            const size_t keep = have / 2 < ((size_t)1 << 30) ? have / 2 : ((size_t)1 << 30);
            size_t fit = (have - keep) / per_proof;
            if (getenv("DOT_RING_B200_DEBUG"))
                fprintf(stderr, "[dot_ring_b200] prove: free %.2f GB (+%.2f GB held), %.2f MB per proof -> up to %zu proofs per pass\n", free_b / 1e9,
                        (double)(have - free_b) / 1e9, per_proof / 1e6, fit);
            if (fit < chunk_cap) chunk_cap = fit < 64 ? 64 : fit;
        }
    }
#endif
    // equal passes: a group of g proofs in ceil(g / cap) passes of the same width (a short last pass would pay the latency-bound
    // kernels again for little work)
    auto pass_width_of = [&](size_t g) {
        const size_t passes = (g + chunk_cap - 1) / chunk_cap;
        return (g + passes - 1) / passes;
    };
    ProveScratch& sc = scratch_for(ctx);
    sc.ensure(pass_width_of(widest), N_max);
    sc.blob.ensure(blob_len ? blob_len : 1);
    h2d(ctx->stream, sc.blob.p, blob, blob_len);
    PhaseTimer& pt = ctx->phases;
    pt.reset();
    pt.active = true;
    struct Deactivate {
        PhaseTimer& p;
        ~Deactivate() { p.active = false; }
    } deactivate{pt};
    std::vector<ProveInput> hin;
    std::vector<uint8_t> hzk, hout;
    std::vector<uint32_t> hstatus;

    for (size_t g = 0, group_begin = 0; g < group_end.size(); group_begin = group_end[g++]) {
        const size_t group_n = group_end[g] - group_begin;
        auto item = [&](size_t j) -> size_t { return direct ? j : order[group_begin + j]; };
        // everything of a pass that depends only on N comes from the group's first ring
        Ring* lead = rings[ring_of(item(0))];
        const RingDev& rg = lead->dev;
        const uint32_t N = rg.N;
        const uint32_t qlen = 3 * N + 1;
        const uint32_t nthr = ntt_threads(N);
        const size_t ntt_smem = ntt_smem_bytes(N);
        const bool large = N > 4096 || ctx->generic_ntt_path;  // two-pass transforms + element-wise twists instead of the fused single-CTA kernels
        const NttPlan* big_plan = large ? &ctx->plan(N, rg.omega) : nullptr;
        const size_t pass_width = pass_width_of(group_n);

        for (size_t base = 0; base < group_n; base += pass_width) {
            const uint32_t m = (uint32_t)((group_n - base < pass_width) ? group_n - base : pass_width);
            pt.mark(ctx, 7);
            hin.assign(m, ProveInput{});
            for (uint32_t i = 0; i < m; i++) {
                const size_t it = item(base + i);
                ProveInput& pi = hin[i];
                if (!bare) {
                    pi.alpha_off = alpha_off[it];
                    pi.alpha_len = alpha_len[it];
                    pi.ad_off = ad_off[it];
                    pi.ad_len = ad_len[it];
                }
                pi.k = producer_index[it];
                pi.ring = ring_of(it);
                memcpy(pi.sk, secrets32 + 32 * it, 32);
            }
            h2d(ctx->stream, sc.in.p, hin.data(), m * sizeof(ProveInput));
            const uint32_t tb = 64, pb = (m + tb - 1) / tb;

            pt.mark(ctx, 0);
            // zk rows (Montgomery) into the state, then Pedersen + witness
            if (zk_rows) {
                const uint8_t* src = zk_rows + base * 12 * 32;
                if (!direct) {
                    hzk.resize((size_t)m * 12 * 32);
                    for (uint32_t i = 0; i < m; i++) memcpy(hzk.data() + (size_t)i * 12 * 32, zk_rows + item(base + i) * 12 * 32, 12 * 32);
                    src = hzk.data();
                }
                h2d(ctx->stream, sc.zraw.p, src, (size_t)m * 12 * 32);
                launch(ctx->stream, Dim3((m * 12 + 127) / 128), 128, 0, ZkRowsBody(), (const uint8_t*)sc.zraw.p, sc.st.p, m);
            } else {
                launch(ctx->stream, Dim3((m * 12 + 127) / 128), 128, 0, ZkRowsBody(), (const uint8_t*)nullptr, sc.st.p, m);
            }
            // Pedersen part: the half the ring proof needs (blinding factor, blinded key) on the main stream, eight lanes per proof; the
            // rest (nonces, R, Ok, responses) on the side stream, joined before the proofs are assembled.  A bare ring proof starts from
            // the caller's blinding factor instead and has no Pedersen part.
            {
                const uint32_t per_block = tb / COOP_LANES;  // eight lanes per proof
                if (bare) {
                    launch(ctx->stream, Dim3((m + per_block - 1) / per_block), tb, ring_proof_start_smem(tb), RingProofStartBody(), suite, dtab, (const ProveInput*)sc.in.p,
                           sc.st.p, m);
                } else {
                    launch(ctx->stream, Dim3((m + per_block - 1) / per_block), tb, pedersen_start_smem(tb), PedersenStartBody(), suite, dtab, (const ProveInput*)sc.in.p,
                           (const uint8_t*)sc.blob.p, sc.st.p, m);
                    ctx->fork_side();
                    launch(ctx->side, Dim3((m + 31) / 32), 32, 0, PedersenFinishBody(), suite, (const ProveInput*)sc.in.p, sc.st.p, m);
                }
            }
            {
                const uint32_t wt = 4 * WIT_LANES;  // four proofs per block, a warp each
                launch(ctx->stream, Dim3((m + 3) / 4), wt, witness_coop_smem(wt), WitnessBody(), rg, dtab, sc.st.p, m);
            }
            pt.mark(ctx, 1);
            // The coefficient form of the witness columns is first needed by the low-degree extension, the commitments by the transcript:
            // on the fused path the interpolation runs on a second side stream next to the (sparse) commitments.
            const bool overlap_intt = !large && !ctx->dense_witness_commit;
            if (!large) {
                if (overlap_intt) ctx->fork_side2();
                launch(overlap_intt ? ctx->side2 : ctx->stream, Dim3(4, m), nthr, ntt_smem, WitnessInttBody(), rg, dtab, (const ProofState*)sc.st.p, sc.wit_coef.p);
            } else {
                launch(ctx->stream, Dim3((N + 127) / 128, 4, m), 128, 0, WitnessEvalBody(), rg, dtab, (const ProofState*)sc.st.p, sc.wit_coef.p);
                ntt_device(ctx, *big_plan, sc.wit_coef.p, sc.wit_coef.p, 4 * (size_t)m, true, sc.ntt_tmp);
            }
            pt.mark(ctx, 2);
            if (ctx->dense_witness_commit || large) {
                commit_device(ctx, lead->srs, sc.wit_coef.p, N, N, 4 * m, sc.res.p);
            } else {
                // the Lagrange table is per SRS and domain: every ring of the group shares it
                const LagrangeTable* lag = lead->lag ? lead->lag : &lead->srs->lagrange_table(N, rg.logN, rg.omega, rg.tw_inv, rg.n_inv);
                for (size_t i = 0; i < m; i++) rings[ring_of(item(base + i))]->lag = lag;
                ctx->partials.ensure((size_t)4 * m);
                launch_lb<64, 8>(ctx->stream, Dim3(4, m), 64, witness_commit_smem(lag->geom.W, 64), WitnessCommitBody(), (const G1Affine*)lag->table.p, lag->geom, rg,
                                 dtab, (const ProofState*)sc.st.p, ctx->partials.p);
                launch_commit_finish(ctx->stream, (const G1*)ctx->partials.p, 1u, 4 * m, sc.res.p);
            }
            // column order (b, accx, accy, accip) -> payload slots (0, 2, 3, 1)
            launch(ctx->stream, Dim3((4 * m + 127) / 128), 128, 0, StoreCommitBody(), (const G1Affine*)sc.res.p, 4u, 0x01030200u, sc.st.p, m);
            pt.mark(ctx, 5);
            launch(ctx->stream, Dim3(pb), tb, 0, Transcript1Body(), sc.st.p, m);
            if (overlap_intt) ctx->join_side2();
            pt.mark(ctx, 3);
            if (!large) {
                launch(ctx->stream, Dim3(16, m), nthr, ntt_smem, WitnessLdeBody(), rg, dtab, (const ProofState*)sc.st.p, (const Fr*)sc.wit_coef.p, sc.lde.p);
            } else {
                launch(ctx->stream, Dim3((N + 127) / 128, 4, 4 * m), 128, 0, CosetTwistBody(), N, rg.w4, (const Fr*)sc.wit_coef.p, sc.lde.p);
                ntt_device(ctx, *big_plan, sc.lde.p, sc.lde.p, 16 * (size_t)m, false, sc.ntt_tmp);
            }
            launch(ctx->stream, Dim3((4 * N + 127) / 128, m), 128, 0, ConstraintBody(), rg, dtab, (const ProofState*)sc.st.p, (const Fr*)sc.lde.p, sc.agg.p);
            if (!large) {
                launch(ctx->stream, Dim3(4, m), nthr, ntt_smem, QuotientInttBody(), rg, sc.agg.p);
            } else {
                ntt_device(ctx, *big_plan, sc.agg.p, sc.agg.p, 4 * (size_t)m, true, sc.ntt_tmp);
                launch(ctx->stream, Dim3((N + 127) / 128, 4, m), 128, 0, CosetUntwistBody(), N, rg.w4inv, sc.agg.p);
            }
            launch(ctx->stream, Dim3((N + 127) / 128, m), 128, 0, QuotientCombineBody(), rg, (const Fr*)sc.agg.p, sc.cagg.p);
            launch(ctx->stream, Dim3((qlen + 127) / 128, m), 128, 0, QuotientFoldBody(), rg, (const Fr*)sc.cagg.p, sc.quot.p, qlen);
            pt.mark(ctx, 2);
            commit_device(ctx, lead->srs, sc.quot.p, qlen, qlen, m, sc.res.p);
            launch(ctx->stream, Dim3((m + 127) / 128), 128, 0, StoreCommitBody(), (const G1Affine*)sc.res.p, 1u, 0x04u, sc.st.p, m);
            pt.mark(ctx, 5);
            launch(ctx->stream, Dim3(pb), tb, 0, Transcript2Body(), sc.st.p, m);
            pt.mark(ctx, 4);
            launch(ctx->stream, Dim3(7, m), 128, 128 * sizeof(Fr), EvalBody(), rg, dtab, sc.st.p, (const Fr*)sc.wit_coef.p);
            launch(ctx->stream, Dim3((N + 127) / 128, m), 128, 0, LinPolyBody(), rg, (const ProofState*)sc.st.p, (const Fr*)sc.wit_coef.p, sc.lin.p);
            launch(ctx->stream, Dim3(1, m), 128, 128 * sizeof(Fr), LinEvalBody(), rg, sc.st.p, (const Fr*)sc.lin.p);
            pt.mark(ctx, 5);
            launch(ctx->stream, Dim3(pb), tb, 0, Transcript3Body(), sc.st.p, m);
            pt.mark(ctx, 4);
            launch(ctx->stream, Dim3((qlen + 127) / 128, m), 128, 0, AggOpenBody(), rg, dtab, (const ProofState*)sc.st.p, (const Fr*)sc.wit_coef.p, (const Fr*)sc.quot.p, qlen,
                   sc.aggopen.p);
            launch(ctx->stream, Dim3(2, m), 256, synthetic_div_smem(256), OpenQuotientsBody(), rg, (const ProofState*)sc.st.p, sc.aggopen.p, qlen, sc.lin.p);
            pt.mark(ctx, 2);
            commit_device_pair(ctx, lead->srs, sc.aggopen.p, qlen, 3 * N, sc.lin.p, N, N - 1, m, sc.res.p);
            launch(ctx->stream, Dim3((m + 127) / 128), 128, 0, StoreCommitBody(), (const G1Affine*)sc.res.p, 1u, 0x05u, sc.st.p, m);
            launch(ctx->stream, Dim3((m + 127) / 128), 128, 0, StoreCommitBody(), (const G1Affine*)(sc.res.p + m), 1u, 0x06u, sc.st.p, m);
            pt.mark(ctx, 5);
            if (bare) {
                launch(ctx->stream, Dim3(pb), tb, 0, RingProofFinalizeBody(), sc.st.p, m, sc.out.p);
            } else {
                ctx->join_side();
                launch(ctx->stream, Dim3(pb), tb, 0, FinalizeBody(), (const ProofState*)sc.st.p, m, sc.out.p, sc.status.p);
            }
            pt.mark(ctx, 8);
            dev_zero(ctx->stream, sc.in.p, m * sizeof(ProveInput));  // secret keys / blinding factors do not outlive the pass on the device
            if (bare && direct) {
                d2h(ctx->stream, res.relations_xy64 + 64 * base, sc.out.p, (size_t)m * 64);
                d2h(ctx->stream, res.payloads592 + 592 * base, sc.out.p + (size_t)m * 64, (size_t)m * 592);
            } else if (direct) {
                d2h(ctx->stream, res.proofs784 + 784 * base, sc.out.p, (size_t)m * 784);
                d2h(ctx->stream, res.status + base, sc.status.p, (size_t)m * sizeof(uint32_t));
            } else {
                hout.resize((size_t)m * 784);
                d2h(ctx->stream, hout.data(), sc.out.p, (size_t)m * (bare ? 656 : 784));
                if (!bare) {
                    hstatus.resize(m);
                    d2h(ctx->stream, hstatus.data(), sc.status.p, (size_t)m * sizeof(uint32_t));
                }
            }
            pt.mark(ctx, -1);
            stream_sync(ctx->stream);
            pt.collect(ctx);
            if (!direct) {
                for (uint32_t i = 0; i < m; i++) {
                    const size_t it = item(base + i);
                    if (bare) {
                        memcpy(res.relations_xy64 + 64 * it, hout.data() + (size_t)64 * i, 64);
                        memcpy(res.payloads592 + 592 * it, hout.data() + (size_t)64 * m + (size_t)592 * i, 592);
                    } else {
                        memcpy(res.proofs784 + 784 * it, hout.data() + (size_t)784 * i, 784);
                        res.status[it] = hstatus[i];
                    }
                }
            }
        }
    }
    {  // ... nor in the host staging buffer (volatile: the stores must not be optimised away)
        volatile uint8_t* w = (volatile uint8_t*)hin.data();
        for (size_t i = 0; i < hin.size() * sizeof(ProveInput); i++) w[i] = 0;
    }
}

// The argument checks dr_ring_prove_multi and dr_ring_proof_prove_multi share: the rings and the ring index.
static void check_prove_rings(Ctx* ctx, Ring* const* rings, size_t n_rings, const uint32_t* ring_index, size_t n) {
    if (n && !n_rings) throw Error(DR_EINVAL, "at least one ring is required");
    for (size_t k = 0; k < n_rings; k++) {
        const Ring* ring = rings[k];
        const Ring* first = rings[0];
        if (!ring) throw Error(DR_EINVAL, "bad argument");
        if (ring->ctx != ctx) throw Error(DR_EINVAL, "ring belongs to another context");
        if (ring->srs != first->srs) throw Error(DR_EINVAL, "rings of one call must share the SRS handle");
        if (!same_suite(ring->suite, first->suite) || !(ring->dev.seed == first->dev.seed) || !(ring->padding == first->padding))
            throw Error(DR_EINVAL, "rings of one call must share the suite");
    }
    // rings of one domain size share its roots of unity: a pass takes the twiddles and coset powers from one of them
    for (size_t k = 0; k < n_rings; k++)
        for (size_t j = 0; j < k; j++)
            if (rings[j]->dev.N == rings[k]->dev.N && (rings[j]->dev.omega != rings[k]->dev.omega || rings[j]->radix_omega != rings[k]->radix_omega))
                throw Error(DR_EINVAL, "rings of one domain size must share omega and radix_omega");
    for (size_t i = 0; i < n; i++)
        if (ring_index[i] >= n_rings) throw Error(DR_EINVAL, "ring index out of range");
}

// ---- ring roots without a ring ----------------------------------------------------------------------------------------------
// What dr_ring_roots_from_keys / dr_ring_root_update read of the params, checked as dr_ring_create checks it, and of the SRS.
struct RootSetup {
    uint32_t N = 0, logN = 0, max_ring = 0;
    Fr omega;
    TEAffine padding, blinding_base;
};

static RootSetup root_setup(Ctx* ctx, Srs* srs, const dr_ring_params* prm) {
    check_ring_shape(prm);
    RootSetup s;
    s.N = prm->domain_size;
    while ((1u << s.logN) < s.N) s.logN++;
    s.max_ring = prm->max_ring_size;
    s.omega = fr_param(prm->omega);
    check_primitive_root(s.omega, s.logN);
    s.padding = te_param(prm->padding_point);
    s.blinding_base = te_param(prm->blinding_base);
    if (srs->ctx != ctx) throw Error(DR_EINVAL, "SRS belongs to another context");
    if (srs->n < s.N) throw Error(DR_EINVAL, "SRS too small for this domain (needs N G1 points)");
    return s;
}

// `batch` evaluation vectors of N elements (in place: -> coefficients) -> their KZG commitments, affine, on the device
static void commit_columns(Ctx* ctx, Srs* srs, const RootSetup& s, Fr* cols, uint32_t batch, G1Affine* out) {
    DevBuf<Fr> ntt_tmp;
    ntt_device(ctx, ctx->plan(s.N, s.omega), cols, cols, batch, true, ntt_tmp);
    commit_device(ctx, srs, cols, s.N, s.N, batch, out);
}

// The root half of dr_ring_create for n_rings key vectors: every ring's px, py and the shared s in one column buffer, one batched
// inverse NTT and one batched commitment per pass.  C_s is committed once, in the first pass.
static void ring_roots(Ctx* ctx, Srs* srs, const RootSetup& s, size_t n_rings, const uint8_t* keys32, const std::vector<uint32_t>& key_off, uint8_t* roots144) {
    const uint32_t N = s.N;
    const size_t total = key_off[n_rings];
    const std::vector<TEAffine> rows = public_vector_rows(N, s.max_ring, s.padding, s.blinding_base);
    DevBuf<TEAffine> drows(N);
    DevBuf<uint8_t> dkeys(total * 32);
    DevBuf<uint32_t> doff(n_rings + 1);
    h2d(ctx->stream, drows.p, rows.data(), N * sizeof(TEAffine));
    h2d(ctx->stream, dkeys.p, keys32, total * 32);
    h2d(ctx->stream, doff.p, key_off.data(), (n_rings + 1) * sizeof(uint32_t));
    // rings per pass: two columns of N elements each, at most 1 GB of columns and 1024 rings (grid rows) at a time
    const size_t by_memory = ((size_t)1 << 30) / (2 * (size_t)N * sizeof(Fr));
    const size_t per_pass = std::min(n_rings, std::min<size_t>(1024, by_memory));
    const uint32_t cap = (uint32_t)(2 * per_pass + 1);
    DevBuf<Fr> cols((size_t)cap * N);
    DevBuf<G1Affine> cm(cap);
    DevBuf<uint8_t> enc(48 * (size_t)cap);
    std::vector<uint8_t> host(48 * (size_t)cap);
    uint8_t c_s[48];
    for (size_t r0 = 0; r0 < n_rings; r0 += per_pass) {
        const uint32_t m = (uint32_t)std::min(per_pass, n_rings - r0);
        const uint32_t with_s = r0 == 0 ? 1 : 0;
        const uint32_t batch = 2 * m + with_s;
        launch(ctx->stream, Dim3((N + 127) / 128, m + with_s), 128, 0, RingRootColumnsBody(), (const TEAffine*)drows.p, (const uint8_t*)dkeys.p,
               (const uint32_t*)(doff.p + r0), m, N, s.max_ring, s.padding, cols.p);
        commit_columns(ctx, srs, s, cols.p, batch, cm.p);
        launch(ctx->stream, Dim3((batch + 63) / 64), 64, 0, G1EncodeBody(), (const G1Affine*)cm.p, batch, (uint8_t*)nullptr, enc.p);
        d2h(ctx->stream, host.data(), enc.p, 48 * (size_t)batch);
        stream_sync(ctx->stream);
        if (with_s) memcpy(c_s, host.data() + 96 * (size_t)m, 48);
        for (uint32_t k = 0; k < m; k++) {
            uint8_t* out = roots144 + 144 * (r0 + k);
            memcpy(out, host.data() + 96 * (size_t)k, 96);
            memcpy(out + 96, c_s, 48);
        }
    }
}

// The root is linear in the column evaluations: C_px' = C_px + commit(iNTT(dx)), dx non-zero on the changed rows only (and py
// alike).  The selector column is committed next to the two differences: the root's C_s must equal it.
static void ring_root_update(Ctx* ctx, Srs* srs, const RootSetup& s, const uint8_t* root144, size_t n, const uint32_t* rows, const uint8_t* old_keys32,
                             const uint8_t* new_keys32, uint8_t* out144) {
    G1Affine in[3];
    for (int i = 0; i < 3; i++)
        if (!g1_decode(in[i], root144 + 48 * i, 48)) throw Error(DR_EINVAL, "invalid BLS12-381 G1 encoding in ring root");
    std::vector<uint8_t> seen(s.max_ring, 0);
    for (size_t j = 0; j < n; j++) {
        if (rows[j] >= s.max_ring) throw Error(DR_EINVAL, "row out of range: key rows lie below max_ring_size");
        if (seen[rows[j]]++) throw Error(DR_EINVAL, "a row appears twice in one update");
    }
    const uint32_t N = s.N;
    DevBuf<Fr> cols(3 * (size_t)N);  // dx | dy | s
    DevBuf<uint8_t> dkeys(2 * n * 32);
    DevBuf<uint32_t> drows(n);
    dev_zero(ctx->stream, cols.p, 2 * (size_t)N * sizeof(Fr));
    if (n) {
        if (old_keys32) h2d(ctx->stream, dkeys.p, old_keys32, n * 32);
        h2d(ctx->stream, dkeys.p + n * 32, new_keys32, n * 32);
        h2d(ctx->stream, drows.p, rows, n * sizeof(uint32_t));
        launch(ctx->stream, Dim3((uint32_t)((n + 63) / 64)), 64, 0, RootDeltaBody(), old_keys32 ? (const uint8_t*)dkeys.p : (const uint8_t*)nullptr,
               (const uint8_t*)(dkeys.p + n * 32), (const uint32_t*)drows.p, (uint32_t)n, N, s.padding, cols.p);
    }
    launch(ctx->stream, Dim3((N + 127) / 128, 1), 128, 0, RingRootColumnsBody(), (const TEAffine*)nullptr, (const uint8_t*)nullptr, (const uint32_t*)nullptr, 0u, N,
           s.max_ring, s.padding, cols.p + 2 * (size_t)N);
    DevBuf<G1Affine> cm(3);
    commit_columns(ctx, srs, s, cols.p, 3, cm.p);
    G1Affine delta[3];
    d2h(ctx->stream, delta, cm.p, sizeof(delta));
    stream_sync(ctx->stream);
    uint8_t c_s[48];
    g1_compress(c_s, delta[2]);
    if (memcmp(c_s, root144 + 96, 48)) throw Error(DR_EINVAL, "ring root does not belong to these params and this SRS (its C_s differs)");
    uint8_t out[144];
    for (int i = 0; i < 2; i++) {
        G1 sum = G1::from_affine(in[i]);
        g1_add(sum, G1::from_affine(delta[i]));
        g1_compress(out + 48 * i, g1_to_affine(sum));
    }
    memcpy(out + 96, c_s, 48);
    memcpy(out144, out, 144);
}

}  // namespace dr

using namespace dr;

extern "C" {

int dr_ring_create(dr_ctx* c, dr_srs* s, const dr_ring_params* prm, const uint8_t* keys32, size_t n_keys, dr_ring** out) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    Srs* srs = (Srs*)s;
    if (!ctx || !srs || !prm || !out || (n_keys && !keys32)) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    const uint32_t N = prm->domain_size;
    check_ring_shape(prm);
    if (n_keys > prm->max_ring_size) throw Error(DR_EINVAL, "ring size exceeds max supported size");
    if (3 * (size_t)N + 1 > srs->n) throw Error(DR_EINVAL, "SRS too small for this domain (needs 3N+1 G1 points)");

    auto ring = std::make_unique<Ring>();
    ring->ctx = ctx;
    ring->srs = srs;
    SuiteDev& su = ring->suite;
    su = suite_param(*prm);
    RingDev& d = ring->dev;
    d.N = N;
    d.logN = 0;
    while ((1u << d.logN) < N) d.logN++;
    const uint32_t max_ring = prm->max_ring_size;
    ring->tab.max_ring = max_ring;
    d.last = N - 4;
    d.omega = fr_param(prm->omega);
    Fr w4 = fr_param(prm->radix_omega);
    ring->radix_omega = w4;
    // sanity: w4^4 == omega, omega^N == 1, omega^(N/2) != 1
    if (w4.sqr().sqr() != d.omega) throw Error(DR_EINVAL, "radix_omega^4 != omega");
    check_primitive_root(d.omega, d.logN);
    d.seed = te_param(prm->seed);
    ring->g_table = ctx->fixed_table(su.generator);
    ring->b_table = ctx->fixed_table(su.blinding_base);
    su.g_tab = ring->g_table->tab.p;
    su.b_tab = ring->b_table->tab.p;
    ring->padding = te_param(prm->padding_point);
    d.n_inv = Fr::from_u32(N).inv();
    d.quarter = Fr::from_u32(4).inv();

    // ---- domain tables (host, portable arithmetic; uploaded once) ----
    const NttPlan& plan = ctx->plan(N, d.omega);
    d.tw_fwd = plan.tw_fwd.p;
    d.tw_inv = plan.tw_inv.p;
    std::vector<Fr> hw4(4 * N), hw4i(4 * N);
    {
        Fr a = Fr::one(), b = Fr::one(), w4i = w4.inv();
        for (uint32_t k = 0; k < 4 * N; k++) {
            hw4[k] = a;
            hw4i[k] = b;
            a = a * w4;
            b = b * w4i;
        }
        if (a != Fr::one()) throw Error(DR_EINVAL, "radix_omega is not a 4N-th root of unity");
    }
    ring->w4.alloc(4 * N);
    ring->w4inv.alloc(4 * N);
    h2d(ctx->stream, ring->w4.p, hw4.data(), 4 * N * sizeof(Fr));
    h2d(ctx->stream, ring->w4inv.p, hw4i.data(), 4 * N * sizeof(Fr));
    d.w4 = ring->w4.p;
    d.w4inv = ring->w4inv.p;
    domain_tail(d.omega, d.tail, d.w_last);

    // ---- public vector PK || padding || 2^i B || zeros (members.py:36-53) ----
    ring->nm.alloc(N);
    {
        std::vector<TEAffine> host = public_vector_rows(N, max_ring, ring->padding, su.blinding_base);
        h2d(ctx->stream, ring->nm.p, host.data(), N * sizeof(TEAffine));
        if (n_keys) {
            DevBuf<uint8_t> kraw(n_keys * 32);
            h2d(ctx->stream, kraw.p, keys32, n_keys * 32);
            launch(ctx->stream, Dim3((uint32_t)((n_keys + 63) / 64)), 64, 0, KeyDecodeBody(), (const uint8_t*)kraw.p, (uint32_t)n_keys, ring->padding, ring->nm.p);
            stream_sync(ctx->stream);
        }
    }
    ring->tab.nm = ring->nm.p;

    // ---- fixed columns: evaluations -> coefficients -> commitments ----
    ring->fixed_coef.alloc(3 * N);
    launch(ctx->stream, Dim3((N + 127) / 128), 128, 0, FixedColumnsBody(), (const TEAffine*)ring->nm.p, N, max_ring, ring->fixed_coef.p);
    const uint32_t nthr = ntt_threads(N);
    DevBuf<Fr> ntt_tmp;
    ntt_device(ctx, plan, ring->fixed_coef.p, ring->fixed_coef.p, 3, true, ntt_tmp);
    ring->tab.fixed_coef = ring->fixed_coef.p;
    DevBuf<G1Affine> cm(3);
    commit_device(ctx, srs, ring->fixed_coef.p, N, N, 3, cm.p);
    DevBuf<uint8_t> enc96(288), enc48(144);
    launch(ctx->stream, Dim3(1), 64, 0, G1EncodeBody(), (const G1Affine*)cm.p, 3u, enc96.p, enc48.p);
    d2h(ctx->stream, ring->commitments, cm.p, 3 * sizeof(G1Affine));
    d2h(ctx->stream, ring->commit_be96, enc96.p, 288);
    d2h(ctx->stream, ring->root144, enc48.p, 144);

    // ---- 4x LDE of px, py, s, L_0, L_{N-4} and (x - w^(N-4)) on the 4N domain ----
    ring->fixed_lde.alloc(6 * 4 * (size_t)N);
    {
        DevBuf<Fr> coef5(5 * (size_t)N);
        d2d(ctx->stream, coef5.p, ring->fixed_coef.p, 3 * N * sizeof(Fr));
        std::vector<Fr> lag(2 * (size_t)N);
        Fr cur0 = d.n_inv, curl = d.n_inv;
        Fr inv_xl = hw4i[4 * (N - 4)];  // w^-(N-4)
        for (uint32_t k = 0; k < N; k++) {
            lag[k] = cur0;  // L_0 = (1/N) sum X^k
            lag[N + k] = curl;
            curl = curl * inv_xl;
        }
        h2d(ctx->stream, coef5.p + 3 * (size_t)N, lag.data(), 2 * N * sizeof(Fr));
        if (N <= 4096 && !ctx->generic_ntt_path) {
            launch(ctx->stream, Dim3(20), nthr, ntt_smem_bytes(N), PlainLdeBody(), N, d.logN, (const Fr*)plan.tw_fwd.p, (const Fr*)ring->w4.p, (const Fr*)coef5.p,
                   ring->fixed_lde.p);
        } else {
            launch(ctx->stream, Dim3((N + 127) / 128, 4, 5), 128, 0, CosetTwistBody(), N, (const Fr*)ring->w4.p, (const Fr*)coef5.p, ring->fixed_lde.p);
            ntt_device(ctx, plan, ring->fixed_lde.p, ring->fixed_lde.p, 20, false, ntt_tmp);
        }
        launch(ctx->stream, Dim3((4 * N + 127) / 128), 128, 0, NotLastBody(), N, (const Fr*)ring->w4.p, d.w_last, ring->fixed_lde.p + 5 * 4 * (size_t)N);
        stream_sync(ctx->stream);
    }
    ring->tab.fixed_lde = ring->fixed_lde.p;

    // ---- verifier key; the prover starts from its transcript prefix under the suite id ----
    ring->vk = make_verifier_key(ctx, N, d.omega, d.seed, su.suite_id, su.suite_id_len, srs->g1_0_be96, srs->g2_be192, ring->commit_be96, ring->vk_lines);
    ring->vk_dev.alloc(1);
    h2d(ctx->stream, ring->vk_dev.p, &ring->vk, sizeof(VerifierKeyDev));
    ring->prefix.alloc(1);
    h2d(ctx->stream, ring->prefix.p, &ring->vk.prefix, sizeof(Shake128));
    ring->tab.prefix = ring->prefix.p;
    ring->tab_dev.alloc(1);
    h2d(ctx->stream, ring->tab_dev.p, &ring->tab, sizeof(RingTab));
    stream_sync(ctx->stream);
    *out = (dr_ring*)ring.release();
    DR_API_END
}

void dr_ring_destroy(dr_ring* r) {
    Ring* ring = (Ring*)r;
    if (!ring) return;
    free_on_owner_stream(ring->ctx);
    delete ring;
}

int dr_ring_root(dr_ring* r, uint8_t root144[144]) {
    DR_API_BEGIN
    if (!r || !root144) throw Error(DR_EINVAL, "bad argument");
    memcpy(root144, ((Ring*)r)->root144, 144);
    DR_API_END
}

int dr_ring_fixed_commitments(dr_ring* r, uint8_t out288[288]) {
    DR_API_BEGIN
    if (!r || !out288) throw Error(DR_EINVAL, "bad argument");
    memcpy(out288, ((Ring*)r)->commit_be96, 288);
    DR_API_END
}

int dr_ring_points(dr_ring* r, uint8_t* out_xy64, size_t n_points) {
    DR_API_BEGIN
    Ring* ring = (Ring*)r;
    if (!ring || !out_xy64 || n_points > ring->dev.N) throw Error(DR_EINVAL, "bad argument");
    ring->ctx->activate();
    std::vector<TEAffine> host(n_points);
    d2h(ring->ctx->stream, host.data(), ring->nm.p, n_points * sizeof(TEAffine));
    stream_sync(ring->ctx->stream);
    for (size_t i = 0; i < n_points; i++) {
        fr_to_le_bytes_raw(out_xy64 + 64 * i, host[i].x.from_mont());
        fr_to_le_bytes_raw(out_xy64 + 64 * i + 32, host[i].y.from_mont());
    }
    DR_API_END
}

int dr_ring_roots_from_keys(dr_ctx* c, dr_srs* s, const dr_ring_params* prm, size_t n_rings, const uint8_t* keys32, const uint32_t* key_counts, uint8_t* roots144) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    Srs* srs = (Srs*)s;
    if (!ctx || !srs || !prm || (n_rings && (!key_counts || !roots144))) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    const RootSetup st = root_setup(ctx, srs, prm);
    std::vector<uint32_t> key_off(n_rings + 1, 0);
    for (size_t k = 0; k < n_rings; k++) {
        if (key_counts[k] > st.max_ring) throw Error(DR_EINVAL, "ring size exceeds max supported size");
        const uint64_t end = (uint64_t)key_off[k] + key_counts[k];
        if (end > UINT32_MAX) throw Error(DR_EINVAL, "more than 2^32 - 1 keys in one call");
        key_off[k + 1] = (uint32_t)end;
    }
    if (key_off[n_rings] && !keys32) throw Error(DR_EINVAL, "bad argument");
    if (!n_rings) return DR_OK;
    ring_roots(ctx, srs, st, n_rings, keys32, key_off, roots144);
    DR_API_END
}

int dr_ring_root_update(dr_ctx* c, dr_srs* s, const dr_ring_params* prm, const uint8_t root144[144], size_t n, const uint32_t* rows, const uint8_t* old_keys32,
                        const uint8_t* new_keys32, uint8_t out_root144[144]) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    Srs* srs = (Srs*)s;
    if (!ctx || !srs || !prm || !root144 || !out_root144 || (n && (!rows || !new_keys32))) throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    const RootSetup st = root_setup(ctx, srs, prm);
    ring_root_update(ctx, srs, st, root144, n, rows, old_keys32, new_keys32, out_root144);
    DR_API_END
}

int dr_ring_prove_batch(dr_ctx* c, dr_ring* r, size_t n, const uint8_t* blob, const uint32_t* alpha_off, const uint32_t* alpha_len, const uint32_t* ad_off,
                        const uint32_t* ad_len, const uint8_t* secret_keys32, const uint32_t* producer_index, const uint8_t* zk_rows, uint8_t* proofs784,
                        uint32_t* status) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    Ring* ring = (Ring*)r;
    if (!ctx || !ring || (n && (!alpha_off || !alpha_len || !ad_off || !ad_len || !secret_keys32 || !producer_index || !proofs784 || !status)))
        throw Error(DR_EINVAL, "bad argument");
    ctx->activate();
    if (!n) return DR_OK;
    ProveOutputs res;
    res.proofs784 = proofs784;
    res.status = status;
    ring_prove(ctx, &ring, ring->tab_dev.p, nullptr, n, blob, alpha_off, alpha_len, ad_off, ad_len, secret_keys32, producer_index, zk_rows, res);
    DR_API_END
}

int dr_ring_prove_multi(dr_ctx* c, dr_ring* const* rs, size_t n_rings, const uint32_t* ring_index, size_t n, const uint8_t* blob, const uint32_t* alpha_off,
                        const uint32_t* alpha_len, const uint32_t* ad_off, const uint32_t* ad_len, const uint8_t* secret_keys32, const uint32_t* producer_index,
                        const uint8_t* zk_rows, uint8_t* proofs784, uint32_t* status) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || (n_rings && !rs) || n_rings > UINT32_MAX ||
        (n && (!ring_index || !alpha_off || !alpha_len || !ad_off || !ad_len || !secret_keys32 || !producer_index || !proofs784 || !status)))
        throw Error(DR_EINVAL, "bad argument");
    Ring* const* rings = (Ring* const*)rs;
    check_prove_rings(ctx, rings, n_rings, ring_index, n);
    ctx->activate();
    if (!n) return DR_OK;
    std::vector<RingTab> table(n_rings);
    for (size_t k = 0; k < n_rings; k++) table[k] = rings[k]->tab;
    DevBuf<RingTab> dtable(n_rings);
    h2d(ctx->stream, dtable.p, table.data(), n_rings * sizeof(RingTab));
    ProveOutputs res;
    res.proofs784 = proofs784;
    res.status = status;
    ring_prove(ctx, rings, dtable.p, ring_index, n, blob, alpha_off, alpha_len, ad_off, ad_len, secret_keys32, producer_index, zk_rows, res);
    DR_API_END
}

int dr_ring_proof_prove_multi(dr_ctx* c, dr_ring* const* rs, size_t n_rings, const uint32_t* ring_index, size_t n, const uint32_t* producer_index,
                              const uint8_t* blinding_le32, const uint8_t* zk_rows, const uint8_t* label, size_t label_len, uint8_t* relations_xy64,
                              uint8_t* payloads592) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || (n_rings && !rs) || n_rings > UINT32_MAX || (label_len && !label) ||
        (n && (!ring_index || !producer_index || !blinding_le32 || !relations_xy64 || !payloads592)))
        throw Error(DR_EINVAL, "bad argument");
    if (label_len > 32) throw Error(DR_EINVAL, "transcript label longer than 32 bytes");
    Ring* const* rings = (Ring* const*)rs;
    check_prove_rings(ctx, rings, n_rings, ring_index, n);
    for (size_t i = 0; i < n; i++) {
        if (producer_index[i] >= rings[ring_index[i]]->tab.max_ring) throw Error(DR_EINVAL, "producer row out of range: rows lie below max_ring_size");
        Fn t;
        for (int j = 0; j < 8; j++) {
            const uint8_t* b = blinding_le32 + 32 * i + 4 * j;
            t.v[j] = (uint32_t)b[0] | (uint32_t)b[1] << 8 | (uint32_t)b[2] << 16 | (uint32_t)b[3] << 24;
        }
        if (!t.is_canonical_raw()) throw Error(DR_EINVAL, "blinding factor is not below the group order");
    }
    ctx->activate();
    if (!n) return DR_OK;
    std::vector<RingTab> table(n_rings);
    for (size_t k = 0; k < n_rings; k++) table[k] = rings[k]->tab;
    // another label than the suite id: one transcript prefix per ring of the call, pointed at by this call's copy of the table
    DevBuf<Shake128> prefixes;
    const SuiteDev& suite = rings[0]->suite;
    if (label_len && !(label_len == suite.suite_id_len && !memcmp(label, suite.suite_id, label_len))) {
        std::vector<Shake128> host(n_rings);
        for (size_t k = 0; k < n_rings; k++)
            host[k] = ring_transcript_prefix(label, (uint32_t)label_len, rings[k]->srs->g1_0_be96, rings[k]->srs->g2_be192, rings[k]->commit_be96);
        prefixes.alloc(n_rings);
        h2d(ctx->stream, prefixes.p, host.data(), n_rings * sizeof(Shake128));
        for (size_t k = 0; k < n_rings; k++) table[k].prefix = prefixes.p + k;
    }
    DevBuf<RingTab> dtable(n_rings);
    h2d(ctx->stream, dtable.p, table.data(), n_rings * sizeof(RingTab));
    ProveOutputs res;
    res.bare = true;
    res.relations_xy64 = relations_xy64;
    res.payloads592 = payloads592;
    ring_prove(ctx, rings, dtable.p, ring_index, n, nullptr, nullptr, nullptr, nullptr, nullptr, blinding_le32, producer_index, zk_rows, res);
    DR_API_END
}

int dr_ring_prove_phase_ms(dr_ctx* c, float out[6]) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || !out) throw Error(DR_EINVAL, "bad argument");
    for (int i = 0; i < 6; i++) out[i] = ctx->phases.total[i];
    if (getenv("DOT_RING_B200_DEBUG"))
        fprintf(stderr, "[dot_ring_b200] prove: copy-in / set-up %.3f ms, copy-out %.3f ms, commit kernel %.3f ms, side stream fork -> done %.3f ms\n", ctx->phases.total[7],
                ctx->phases.total[8], ctx->phases.total[6], ctx->side_span_ms());
    DR_API_END
}

int dr_ring_prove_commit_kernel_ms(dr_ctx* c, float* ms, uint32_t* launches) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx || !ms || !launches) throw Error(DR_EINVAL, "bad argument");
    *ms = ctx->phases.total[6];
    *launches = ctx->phases.kernel_launches;
    DR_API_END
}

uint32_t dr_ring_witness_table_bits(const dr_ring* r) {
    const Ring* ring = (const Ring*)r;
    return ring && ring->lag ? ring->lag->geom.c : 0;
}

int dr_ctx_set_generic_ntt_path(dr_ctx* c, int enabled) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx) throw Error(DR_EINVAL, "bad argument");
    ctx->generic_ntt_path = enabled != 0;
    DR_API_END
}

int dr_ctx_set_dense_witness_commit(dr_ctx* c, int enabled) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx) throw Error(DR_EINVAL, "bad argument");
    ctx->dense_witness_commit = enabled != 0;
    DR_API_END
}

int dr_ctx_set_prove_chunk(dr_ctx* c, size_t chunk) {
    DR_API_BEGIN
    Ctx* ctx = (Ctx*)c;
    if (!ctx) throw Error(DR_EINVAL, "bad argument");
    ctx->prove_chunk = chunk;
    DR_API_END
}

}  // extern "C"
