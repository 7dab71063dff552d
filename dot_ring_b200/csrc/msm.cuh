// KZG commitments over the fixed G1 SRS: fixed-base window tables in HBM + batched commit kernel.
//
// The reference commits with blst's single-threaded Pippenger over the SRS prefix
// (dot_ring/ring_proof/pcs/kzg.py:152-175, `mult_pippenger(srs.blst_g1_memory[:len], coeffs)`),
// seven times per proof (4 witness columns, quotient, two openings; proof_builder.py:38-142).
// Here every one of those MSMs uses the same bases, so the bases are expanded ONCE per SRS into a
// table  T[i][w][d-1] = d * 2^(c*w) * [tau^i]_1   (d = 1 .. 2^(c-1), affine, Montgomery)
// that lives in HBM (c = 12: 6145 * 22 * 2048 * 96 B = 26.6 GB of the 180 GB), and a commitment is
// just  sum_i sum_w  +-T[i][w][|digit_w(k_i)|]  : W mixed additions per coefficient, no buckets, no
// sort, no doublings, perfectly balanced across threads.  The group element is identical to what
// Pippenger returns, so the commitment bytes are identical.
#pragma once
#include "g1.cuh"
#include "rt.cuh"

namespace dr {

// ---- GLV: k = k1 + k2 * lambda (mod r), lambda = x^2 - 1 (x the BLS12-381 parameter), lambda^2 + lambda + 1 = r, and
// lambda * (X, Y) = (beta * X, Y) on G1.  k2 = floor(k / lambda), k1 = k mod lambda; both are below 2^128, so a table that
// covers 128 bits serves both halves: sum_i k_i P_i = A + phi(B) with A, B accumulated from the same entries.
#define DR_GLV_LAMBDA {0xffffffffu, 0x00000000u, 0x0001a402u, 0xac45a401u}
#define DR_GLV_MU {0xf6cfee30u, 0x63f6e522u, 0xe01faaddu, 0x7c6becf1u, 0x1u} /* floor(2^256 / lambda) */
DR_HD Fq glv_beta() {  // Montgomery form of the cube root of unity matching lambda
    Fq b;
    constexpr uint32_t m[12] = {0x8671f071u, 0xcd03c9e4u, 0x1fcda5d2u, 0x5dab2246u, 0xd3851b95u, 0x587042afu,
                                0x01bacb9eu, 0x8eb60ebeu, 0x83d050d2u, 0x03f97d6eu, 0x54638741u, 0x18f02065u};
    for (int i = 0; i < 12; i++) b.v[i] = m[i];
    return b;
}
// k: 8 canonical limbs (< r).  out: the selected half (which == 0: k1, else k2) as 8 limbs, upper four zero.
DR_HD void glv_half(const uint32_t* k, uint32_t which, uint32_t* out) {
    constexpr uint32_t GLV_LAMBDA[4] = DR_GLV_LAMBDA;
    constexpr uint32_t GLV_MU[5] = DR_GLV_MU;
    // q = (k * mu) >> 256 (Barrett): never above floor(k / lambda) and at most one below it
    uint32_t prod[13];
    for (int i = 0; i < 13; i++) prod[i] = 0;
    for (int i = 0; i < 8; i++) {
        uint64_t carry = 0;
        for (int j = 0; j < 5; j++) {
            uint64_t t = (uint64_t)k[i] * GLV_MU[j] + prod[i + j] + carry;
            prod[i + j] = (uint32_t)t;
            carry = t >> 32;
        }
        prod[i + 5] = (uint32_t)carry;
    }
    uint32_t q[5] = {prod[8], prod[9], prod[10], prod[11], prod[12]};  // q <= lambda + 1 < 2^128: q[4] == 0
    // rem = k - q * lambda, at most 2 * lambda: five limbs are enough
    uint32_t ql[8];
    for (int i = 0; i < 8; i++) ql[i] = 0;
    for (int i = 0; i < 4; i++) {
        uint64_t carry = 0;
        for (int j = 0; j < 4; j++) {
            uint64_t t = (uint64_t)q[i] * GLV_LAMBDA[j] + ql[i + j] + carry;
            ql[i + j] = (uint32_t)t;
            carry = t >> 32;
        }
        ql[i + 4] = (uint32_t)carry;
    }
    uint32_t rem[5];
    uint64_t borrow = 0;
    for (int i = 0; i < 5; i++) {
        uint64_t t = (uint64_t)k[i] - ql[i] - borrow;
        rem[i] = (uint32_t)t;
        borrow = (t >> 32) & 1;
    }
    // rem >= lambda ?  (rem[4] != 0, or the low four limbs compare >=)
    bool ge = rem[4] != 0;
    if (!ge) {
        ge = true;
        for (int i = 3; i >= 0; i--) {
            if (rem[i] != GLV_LAMBDA[i]) {
                ge = rem[i] > GLV_LAMBDA[i];
                break;
            }
        }
    }
    if (ge) {
        borrow = 0;
        for (int i = 0; i < 5; i++) {
            uint64_t t = (uint64_t)rem[i] - (i < 4 ? GLV_LAMBDA[i] : 0u) - borrow;
            rem[i] = (uint32_t)t;
            borrow = (t >> 32) & 1;
        }
        uint64_t carry = 1;
        for (int i = 0; i < 5; i++) {
            uint64_t t = (uint64_t)q[i] + carry;
            q[i] = (uint32_t)t;
            carry = t >> 32;
        }
    }
    for (int i = 0; i < 4; i++) out[i] = which ? q[i] : rem[i];
    for (int i = 4; i < 8; i++) out[i] = 0;
}

// G1 membership (Scott, ePrint 2021/1130): a point P of E(Fq) lies in G1 iff [x^2]P == -phi^2(P) = (beta^2 X, -Y), with
// beta^2 = -1 - beta.  Decoding checks no subgroup (blst's P1_Affine(bytes) does not), and k1 * P + k2 * phi(P) equals k * P only
// on G1: the verifier sends the points that fail this test down a plain full-scalar path, so every curve point gets blst's k * P.
DR_HD_COLD G1 g1_mul_abs_x(const G1& p) {  // [|x|]P, |x| = 0xd201000000010000
    G1 acc = p;
#pragma unroll 1
    for (int bit = 62; bit >= 0; bit--) {
        acc = g1_dbl(acc);
        if ((0xd201000000010000ull >> bit) & 1) g1_add(acc, p);
    }
    return acc;
}
DR_HD_COLD bool g1_in_subgroup(const G1Affine& a) {
    if (a.is_inf()) return true;
    const G1 t = g1_mul_abs_x(g1_mul_abs_x(G1::from_affine(a)));
    if (t.is_inf()) return false;
    const Fq b2x = (a.x + a.x * glv_beta()).neg();
    return t.X == b2x * t.ZZ && t.Y == a.y.neg() * t.ZZZ;
}

struct TableGeom {
    uint32_t c;        // bits of a (narrow) window
    uint32_t W;        // windows; W * c + wide >= 256 (128 with glv)
    uint32_t H;        // entries per (i, w) of a narrow window = 2^(c-1)
    uint32_t n_points; // SRS points covered
    uint32_t wide;     // the `wide` lowest windows take c + 1 bits (2H entries each): one window fewer per scalar for (W + wide) / (W + 1)
                       // of the memory; 0 = uniform windows
    uint32_t glv;      // the table covers 128 bits and every scalar is split in two halves (2W additions per coefficient)
    uint32_t top;      // entries of the last window when it has to hold more than its signed range (glv: the halves run up to
                       // lambda + 1, whose top digit can exceed H); 0 = like any other window
    DR_HD uint32_t width(uint32_t w) const { return c + (w < wide ? 1u : 0u); }
    DR_HD uint32_t bit(uint32_t w) const { return w * c + (w < wide ? w : wide); }
    DR_HD uint32_t entries(uint32_t w) const { return (top && w + 1 == W) ? top : (w < wide ? 2 * H : H); }
    DR_HD uint32_t max_entries() const {
        uint32_t m = wide ? 2 * H : H;
        return top > m ? top : m;
    }
    DR_HD uint32_t additions() const { return glv ? 2 * W : W; }
    // point i owns per_point() consecutive entries; window w starts at (w + min(w, wide)) * H (the last window may be longer)
    DR_HD size_t per_point() const { return ((size_t)(W + wide) << (c - 1)) + (top ? top - entries_plain(W - 1) : 0); }
    DR_HD uint32_t entries_plain(uint32_t w) const { return w < wide ? 2 * H : H; }
    DR_HD size_t entry(uint32_t i, uint32_t w, uint32_t d) const { return (size_t)i * per_point() + ((size_t)(w + (w < wide ? w : wide)) << (c - 1)) + (d - 1); }
    size_t total_entries() const { return (size_t)n_points * per_point(); }
};
inline TableGeom make_geom(uint32_t c, uint32_t n_points, uint32_t wide = 0, uint32_t glv = 0) {
    TableGeom g;
    g.c = c;
    const uint32_t bits = glv ? 128 : 256;
    g.W = (bits - wide + c - 1) / c;
    g.H = 1u << (c - 1);
    g.n_points = n_points;
    g.wide = wide;
    g.glv = glv;
    g.top = 0;
    if (glv) {
        constexpr uint32_t GLV_LAMBDA[4] = DR_GLV_LAMBDA;
        // largest top digit: (lambda + 1) >> bit(W - 1), plus the carry of the window below
        const uint32_t b = g.bit(g.W - 1);
        uint64_t hi = ((uint64_t)GLV_LAMBDA[3] << 32) | GLV_LAMBDA[2];  // bits 64..127 of lambda
        uint64_t top_digit = b >= 64 ? hi >> (b - 64) : ~(uint64_t)0;
        uint64_t need = top_digit + 2;
        if (need > g.entries_plain(g.W - 1)) g.top = (uint32_t)need;
    }
    return g;
}

// ---- SRS ingestion: 96-byte big-endian uncompressed points -> Montgomery affine --------------------
struct SrsLoadBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* in, G1Affine* out, uint32_t n, uint32_t* bad) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < n) {
                G1Affine a;
                if (!g1_decode(a, in + 96 * (size_t)i, 96) || a.is_inf()) {
                    *bad = 1;
                    a = G1Affine::inf();
                }
                out[i] = a;
            }
        }
    }
};

// ---- table construction -------------------------------------------------------------------------
// A thread builds, for one SRS point, R = MAXW / W runs of L consecutive digits in every window: R * W chains E <- E + B_w that
// advance in lockstep, so that each step's affine additions share one field inversion (Montgomery's trick).  Window w holds the
// digits 1..entries(w); chains whose digit has passed that bound simply drop out of the batch.
template <int MAXW>
struct TableBuildBody {
    DR_HD void operator()(const BlockCtx& ctx, const G1Affine* srs, G1Affine* table, TableGeom g, uint32_t chunks) const {
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t W = g.W;
            const uint32_t R = (uint32_t)MAXW / W ? (uint32_t)MAXW / W : 1;  // runs per thread
            const uint32_t groups = (chunks + R - 1) / R;
            const uint32_t gid = ctx.bx * ctx.nthreads + t;
            const uint32_t i = gid / groups, q0 = (gid % groups) * R;
            const uint32_t max_e = g.max_entries();
            const uint32_t L = (max_e + chunks - 1) / chunks;
            if (i < g.n_points && q0 * L + 1 <= max_e) {
                const uint32_t lanes = R * W;  // lane l = r * W + w: run r of window w, first digit (q0 + r) * L + 1
                Fq bx[MAXW], by[MAXW], ex[MAXW], ey[MAXW], den[MAXW], pre[MAXW];
                // 1. window bases B_w = 2^bit(w) * P_i
                {
                    G1 cur = G1::from_affine(srs[i]);
                    G1 proj[MAXW];
#pragma unroll 1
                    for (uint32_t w = 0; w < W; w++) {
                        proj[w] = cur;
                        if (w + 1 < W)
#pragma unroll 1
                            for (uint32_t k = 0; k < g.width(w); k++) cur = g1_dbl(cur);
                    }
                    // batch normalise: x = X / ZZ, y = Y / ZZZ
                    Fq acc = Fq::one();
#pragma unroll 1
                    for (uint32_t w = 0; w < W; w++) {
                        pre[w] = acc;
                        den[w] = proj[w].ZZ * proj[w].ZZZ;
                        acc = acc * den[w];
                    }
                    Fq inv = acc.inv();
#pragma unroll 1
                    for (int w = (int)W - 1; w >= 0; w--) {
                        Fq di = inv * pre[w];
                        inv = inv * den[w];
                        bx[w] = proj[w].X * (di * proj[w].ZZZ);
                        by[w] = proj[w].Y * (di * proj[w].ZZ);
                    }
                }
                // 2. run starts E_l = d0(l) * B_w
                {
                    G1 proj[MAXW];
#pragma unroll 1
                    for (uint32_t l = 0; l < lanes; l++) {
                        const uint32_t w = l % W, d0 = (q0 + l / W) * L + 1;
                        if (d0 > g.entries(w)) continue;
                        G1Affine b{bx[w], by[w]};
                        G1 acc = G1::inf();
#pragma unroll 1
                        for (int bit = 31; bit >= 0; bit--) {
                            acc = g1_dbl(acc);
                            if ((d0 >> bit) & 1) g1_madd(acc, b);
                        }
                        proj[l] = acc;
                    }
                    Fq acc = Fq::one();
#pragma unroll 1
                    for (uint32_t l = 0; l < lanes; l++) {
                        pre[l] = acc;
                        if ((q0 + l / W) * L + 1 > g.entries(l % W)) continue;
                        den[l] = proj[l].ZZ * proj[l].ZZZ;
                        acc = acc * den[l];
                    }
                    Fq inv = acc.inv();
#pragma unroll 1
                    for (int l = (int)lanes - 1; l >= 0; l--) {
                        const uint32_t w = (uint32_t)l % W, d0 = (q0 + (uint32_t)l / W) * L + 1;
                        if (d0 > g.entries(w)) continue;
                        Fq di = inv * pre[l];
                        inv = inv * den[l];
                        ex[l] = proj[l].X * (di * proj[l].ZZZ);
                        ey[l] = proj[l].Y * (di * proj[l].ZZ);
                        table[g.entry(i, w, d0)] = G1Affine{ex[l], ey[l]};
                    }
                }
                // 3. E_l += B_w, one shared inversion per step
#pragma unroll 1
                for (uint32_t o = 1; o < L; o++) {
                    Fq acc = Fq::one();
                    uint32_t active = 0;
#pragma unroll 1
                    for (uint32_t l = 0; l < lanes; l++) {
                        pre[l] = acc;
                        const uint32_t w = l % W, d = (q0 + l / W) * L + 1 + o;
                        if (d > g.entries(w)) continue;
                        // E == B only for d == 2 (then the chord degenerates to the tangent); E == -B never
                        den[l] = (d == 2) ? ey[l].dbl() : bx[w] - ex[l];
                        acc = acc * den[l];
                        active++;
                    }
                    if (!active) break;
                    Fq inv = acc.inv();
#pragma unroll 1
                    for (int l = (int)lanes - 1; l >= 0; l--) {
                        const uint32_t w = (uint32_t)l % W, d = (q0 + (uint32_t)l / W) * L + 1 + o;
                        if (d > g.entries(w)) continue;
                        Fq di = inv * pre[l];
                        inv = inv * den[l];
                        Fq num;
                        if (d == 2) {
                            Fq xx = ex[l].sqr();
                            num = xx.dbl() + xx;
                        } else {
                            num = by[w] - ey[l];
                        }
                        Fq lam = num * di;
                        Fq x3 = lam.sqr() - ex[l] - bx[w];
                        Fq y3 = lam * (ex[l] - x3) - ey[l];
                        ex[l] = x3;
                        ey[l] = y3;
                        table[g.entry(i, w, d)] = G1Affine{x3, y3};
                    }
                }
            }
        }
    }
};

// ---- Lagrange prefix-sum bases ------------------------------------------------------------------------------
// [L_i(tau)]_1 = (1/N) sum_k w^(-ik) [tau^k]_1 is an inverse DFT over group elements: log2 N radix-2 stages of N/2
// butterflies (one scalar multiplication each), then S_j = sum_{i<j} [L_i(tau)]_1.  One-off per (SRS, domain).
struct G1BitReverseBody {  // out[rev(i)] = in[i]
    DR_HD void operator()(const BlockCtx& ctx, const G1Affine* in, uint32_t N, uint32_t logN, G1* out) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < N) {
                uint32_t r = 0;
                for (uint32_t b = 0; b < logN; b++) r |= ((i >> b) & 1u) << (logN - 1 - b);
                out[r] = G1::from_affine(in[i]);
            }
        }
    }
};
// stage with butterfly span `half`: (a, b) -> (a + w b, a - w b), w = winv_half[(N / (2 half)) * j]
struct G1NttStageBody {
    DR_HD void operator()(const BlockCtx& ctx, G1* data, uint32_t N, uint32_t half, const Fr* winv_half) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < N / 2) {
                uint32_t j = i % half, base = (i / half) * 2 * half + j;
                G1 a = data[base], b = data[base + half];
                if (j) {
                    Fr w = winv_half[(N / (2 * half)) * j].from_mont();
                    b = g1_mul_limbs(b, w.v);
                }
                G1 s = a;
                g1_add(s, b);
                g1_add(a, g1_neg(b));
                data[base] = s;
                data[base + half] = a;
            }
        }
    }
};
// data[i] <- (1/N) data[i]
struct G1ScaleBody {
    DR_HD void operator()(const BlockCtx& ctx, G1* data, uint32_t N, Fr n_inv) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < N) {
                Fr k = n_inv.from_mont();
                data[i] = g1_mul_limbs(data[i], k.v);
            }
        }
    }
};
// inclusive prefix sums in place, then affine: out[j-1] = S_j = sum_{i<j} data[i], j = 1..N.  One block, two phases.
struct G1PrefixSumBody {
    DR_HD void operator()(const BlockCtx& ctx, G1* data, uint32_t N, G1Affine* out) const {
        G1* sm = (G1*)ctx.smem;  // per-thread chunk totals
        const uint32_t per = (N + ctx.nthreads - 1) / ctx.nthreads;
        DR_THREAD_LOOP(t, ctx) {
            G1 acc = G1::inf();
            uint32_t lo = t * per, hi = lo + per < N ? lo + per : N;
#pragma unroll 1
            for (uint32_t i = lo; i < hi; i++) {
                g1_add(acc, data[i]);
                data[i] = acc;
            }
            sm[t] = acc;
        }
        DR_BLOCK_SYNC();
        DR_THREAD_LOOP(t, ctx) {
            G1 off = G1::inf();
#pragma unroll 1
            for (uint32_t u = 0; u < t; u++) g1_add(off, sm[u]);
            uint32_t lo = t * per, hi = lo + per < N ? lo + per : N;
#pragma unroll 1
            for (uint32_t i = lo; i < hi; i++) {
                G1 v = data[i];
                g1_add(v, off);
                out[i] = g1_to_affine(v);
            }
        }
    }
};

// ---- signed-digit recoding -------------------------------------------------------------------------
// k: canonical little-endian limbs (< 2^255).  Returns digit w in [-(H-1), H]; carry is threaded.
// `H`: largest digit the window stores (2^(c-1) for a signed window)
DR_HD int msm_digit(const uint32_t* k, uint32_t bit, uint32_t c, uint32_t H, uint32_t& carry) {
    uint32_t limb = bit >> 5, off = bit & 31;
    uint64_t two = (limb < 8 ? (uint64_t)k[limb] : 0) | ((limb + 1 < 8 ? (uint64_t)k[limb + 1] : 0) << 32);
    uint32_t raw = (uint32_t)(two >> off) & ((1u << c) - 1);
    uint32_t d = raw + carry;
    if (d > H) {
        carry = 1;
        return (int)d - (int)(1u << c);
    }
    carry = 0;
    return (int)d;
}
DR_HD int msm_digit(const uint32_t* k, uint32_t w, const TableGeom& g, uint32_t& carry) { return msm_digit(k, g.bit(w), g.width(w), g.entries(w), carry); }
// uniform windows of c bits
DR_HD int msm_digit(const uint32_t* k, uint32_t w, uint32_t c, uint32_t& carry) { return msm_digit(k, w * c, c, 1u << (c - 1), carry); }

// ---- batched commit ----------------------------------------------------------------------------------
// grid = (slices, batch).  MSM `by` uses scalars[by * scalar_stride + i] (Montgomery Fr), i < n, against
// SRS points 0..n-1.  Each block accumulates its slice of points and tree-reduces to one XYZZ partial.
template <bool GLV>
struct CommitBodyT {
    // keep: how many partial sums a CTA leaves (a power of two <= nthreads).  1 = the CTA folds itself completely (large batches:
    // one slice per polynomial, the tree is ~1 % of a CTA's life); 32 = the tree stops after the cross-warp levels and the finish
    // kernel folds the rest (sliced launches of small batches: a full 7-level tree of dependent additions, with three of four
    // warps idle, was ~6 % of a CTA's life there).  partials[(by * slices + bx) * keep + t].
    DR_HD void operator()(const BlockCtx& ctx, const G1Affine* table, TableGeom g, const Fr* scalars, size_t scalar_stride, uint32_t n, G1* partials, uint32_t keep) const {
        G1* sm = (G1*)ctx.smem;
        const uint32_t slices = ctx.gx;
        const uint32_t per = (n + slices - 1) / slices;
        const uint32_t lo = ctx.bx * per;
        const uint32_t hi = (lo + per < n) ? lo + per : n;
        const Fr* sc = scalars + (size_t)ctx.by * scalar_stride;
        DR_THREAD_LOOP(t, ctx) {
            // with a GLV table: pass 0 sums the entries selected by the k1 halves, pass 1 those of the k2 halves; the endomorphism
            // is applied once to the second sum (phi is a homomorphism), so each pass is the plain loop over a 128-bit scalar
#pragma unroll 1
            for (uint32_t pass = 0; pass < (GLV ? 2u : 1u); pass++) {
                G1 acc = G1::inf();
#pragma unroll 1
                for (uint32_t i = lo + t; i < hi; i += ctx.nthreads) {
                    Fr kc = sc[i].from_mont();
                    if (GLV) {
                        uint32_t half[8];
                        glv_half(kc.v, pass, half);
                        for (int l = 0; l < 8; l++) kc.v[l] = half[l];
                    }
                    uint32_t carry = 0;
                    int d_next = msm_digit(kc.v, 0, g, carry);
                    G1Affine pt_next = G1Affine::inf();
                    if (d_next) pt_next = table[g.entry(i, 0, (uint32_t)(d_next < 0 ? -d_next : d_next))];
#pragma unroll 1
                    for (uint32_t w = 0; w < g.W; w++) {
                        int d = d_next;
                        G1Affine pt = pt_next;
                        if (w + 1 < g.W) {
                            d_next = msm_digit(kc.v, w + 1, g, carry);
                            if (d_next) pt_next = table[g.entry(i, w + 1, (uint32_t)(d_next < 0 ? -d_next : d_next))];
                        }
                        if (d) g1_madd(acc, pt, d < 0);
                    }
                }
                if (GLV && pass) {
                    acc.X = acc.X * glv_beta();
                    g1_add(acc, sm[t]);
                }
                sm[t] = acc;
            }
        }
        DR_BLOCK_SYNC();
        for (uint32_t stride = ctx.nthreads >> 1; stride >= keep; stride >>= 1) {
            DR_STRIDE_LOOP(t, stride, ctx) {
                G1 a = sm[t];
                g1_add(a, sm[t + stride]);
                sm[t] = a;
            }
            DR_BLOCK_SYNC();
        }
        DR_THREAD_LOOP(t, ctx) {
            if (t < keep) partials[((size_t)ctx.by * slices + ctx.bx) * keep + t] = sm[t];
        }
    }
};

using CommitBody = CommitBodyT<false>;
using CommitGlvBody = CommitBodyT<true>;

// ---- batched-affine commit --------------------------------------------------------------------------------
// Same sum as CommitBody, cheaper additions.  Adding two affine points costs 2M + 1S once 1/(x2 - x1) is known, and
// Montgomery's trick turns P inversions into one inversion + 3(P - 1) multiplications, so a round that adds P independent
// pairs costs 6 multiplications per addition + 570 / P for the one Fermat inversion, against 10 for an XYZZ mixed addition.
// The table entries one lane must sum (its points x W windows, ~3.6 k for a 6145-coefficient polynomial over 32 lanes) are
// independent, so the lane sums them as a binary tree: round 1 pairs table entries, round k pairs the results of round
// k - 1 (ping-pong buffers in HBM scratch), and once fewer than AFFINE_MIN_PAIRS pairs remain the rest is accumulated in XYZZ
// coordinates as before.  One warp per polynomial; a persistent grid of CTAs walks the batch so that the scratch is per
// resident lane.  All exceptional cases of the affine law (infinity operands, P == Q, P == -Q) are exact: the denominator is
// replaced by 2y (doubling) or 1 (no arithmetic needed) so that they share the batch inversion.
constexpr uint32_t AFFINE_MIN_PAIRS = 160;

struct AffineScratch {  // per lane, interleaved by lane within the warp: element j of lane l at [j * 32 + l]
    uint32_t* refs;     // table entry | sign << 31
    Fq* prefix;
    G1Affine* buf_a;
    G1Affine* buf_b;
    uint32_t cap_refs;  // per lane
};

DR_HD Fq affine_pair_den(const G1Affine& P, const G1Affine& Q) {
    if (P.is_inf() || Q.is_inf()) return Fq::one();
    Fq dx = Q.x - P.x;
    if (!dx.is_zero()) return dx;
    if (P.y == Q.y) return P.y.dbl();  // doubling: lambda = 3 x^2 / (2 y); y != 0 in a prime-order group
    return Fq::one();                  // P == -Q
}
DR_HD G1Affine affine_pair_sum(const G1Affine& P, const G1Affine& Q, const Fq& dinv) {
    if (P.is_inf()) return Q;
    if (Q.is_inf()) return P;
    Fq dx = Q.x - P.x;
    Fq lam;
    if (!dx.is_zero()) {
        lam = (Q.y - P.y) * dinv;
    } else if (P.y == Q.y) {
        Fq xx = P.x.sqr();
        lam = (xx.dbl() + xx) * dinv;
    } else {
        return G1Affine::inf();
    }
    Fq x3 = lam.sqr() - P.x - Q.x;
    return {x3, lam * (P.x - x3) - P.y};
}

// out[i] = in(2i) + in(2i + 1) for i < pairs, one inversion for the whole round.  The first sweep needs only the x
// coordinates (the rare x1 == x2 / x == 0 cases reload the full points); both sweeps fetch the next pair before they use
// the current one so that the gathers overlap the multiplications.
template <class Load, class LoadX>
DR_HD void affine_round(uint32_t pairs, uint32_t lane, const Load& load, const LoadX& load_x, Fq* prefix, G1Affine* out) {
    Fq acc = Fq::one();
    Fq nx1 = load_x(0), nx2 = load_x(1);
#pragma unroll 1
    for (uint32_t i = 0; i < pairs; i++) {
        Fq x1 = nx1, x2 = nx2;
        if (i + 1 < pairs) {
            nx1 = load_x(2 * i + 2);
            nx2 = load_x(2 * i + 3);
        }
        Fq den = x2 - x1;
        if (den.is_zero() || x1.is_zero() || x2.is_zero()) den = affine_pair_den(load(2 * i), load(2 * i + 1));  // exact exceptional cases
        prefix[(size_t)i * 32 + lane] = acc;
        acc = acc * den;
    }
    Fq inv = acc.inv();
    G1Affine nP = load(2 * (pairs - 1)), nQ = load(2 * (pairs - 1) + 1);
#pragma unroll 1
    for (uint32_t i = pairs; i-- > 0;) {
        G1Affine P = nP, Q = nQ;
        if (i > 0) {
            nP = load(2 * i - 2);
            nQ = load(2 * i - 1);
        }
        Fq dinv = inv * prefix[(size_t)i * 32 + lane];
        inv = inv * affine_pair_den(P, Q);
        out[(size_t)i * 32 + lane] = affine_pair_sum(P, Q, dinv);
    }
}

// grid = persistent CTAs; block = warps_per_cta x 32 lanes.  Work item = (polynomial, slice): the points of a polynomial are
// dealt to `slices` warps (point i belongs to lane i % 32 of slice (i / 32) % slices), so that small batches still fill the
// machine.  Warp `wq` of CTA `bx` owns scratch slot bx * warps + wq and walks the work items slot, slot + total_slots, ...
// partials[msm * slices + slice] = XYZZ sum (CommitFinishBody with `slices` follows).
struct CommitAffineBody {
    DR_HD void operator()(const BlockCtx& ctx, const G1Affine* table, TableGeom g, const Fr* scalars, size_t scalar_stride, uint32_t n, uint32_t batch,
                          uint32_t slices, AffineScratch sc, G1* partials) const {
        G1* sm = (G1*)ctx.smem;  // nthreads entries
        const uint32_t warps = ctx.nthreads / 32;
        const uint32_t total_slots = ctx.gx * warps;
        const uint32_t items = batch * slices;
        const uint32_t sweeps = (items + total_slots - 1) / total_slots;
        for (uint32_t it = 0; it < sweeps; it++) {
            DR_THREAD_LOOP(t, ctx) {
                const uint32_t wq = t / 32, lane = t % 32;
                const uint32_t slot = ctx.bx * warps + wq;
                const uint32_t item = it * total_slots + slot;
                G1 acc = G1::inf();
                if (item < items) {
                    const uint32_t msm = item / slices, slice = item % slices;
                    const size_t base = (size_t)slot * sc.cap_refs * 32;
                    uint32_t* refs = sc.refs + base;
                    Fq* prefix = sc.prefix + base / 2;
                    G1Affine* buf_a = sc.buf_a + base / 2;
                    G1Affine* buf_b = sc.buf_b + base / 4;
                    const Fr* sv = scalars + (size_t)msm * scalar_stride;
                    // 1. table references of this lane's points
                    uint32_t count = 0;
#pragma unroll 1
                    for (uint32_t i = slice * 32 + lane; i < n; i += 32 * slices) {
                        Fr kc = sv[i].from_mont();
                        uint32_t carry = 0;
#pragma unroll 1
                        for (uint32_t w = 0; w < g.W; w++) {
                            int d = msm_digit(kc.v, w, g, carry);
                            if (d) {
                                refs[(size_t)count * 32 + lane] = (uint32_t)g.entry(i, w, (uint32_t)(d < 0 ? -d : d)) | (d < 0 ? 0x80000000u : 0u);
                                count++;
                            }
                        }
                    }
                    auto load_ref = [&](uint32_t j) {
                        uint32_t r = refs[(size_t)j * 32 + lane];
                        G1Affine a = table[r & 0x7FFFFFFFu];
                        if (r >> 31) a.y = a.y.neg();
                        return a;
                    };
                    auto load_ref_x = [&](uint32_t j) { return table[refs[(size_t)j * 32 + lane] & 0x7FFFFFFFu].x; };
                    // 2. pairing rounds; an odd element out goes straight to the accumulator
                    uint32_t level = 0;
                    G1Affine* cur = nullptr;
                    while (count / 2 >= AFFINE_MIN_PAIRS) {
                        const uint32_t pairs = count / 2;
                        G1Affine* dst = (level & 1) ? buf_b : buf_a;
                        if (level == 0) {
                            if (count & 1) g1_madd(acc, load_ref(count - 1));
                            affine_round(pairs, lane, load_ref, load_ref_x, prefix, dst);
                        } else {
                            const G1Affine* src = cur;
                            auto load_buf = [&](uint32_t j) { return src[(size_t)j * 32 + lane]; };
                            auto load_buf_x = [&](uint32_t j) { return src[(size_t)j * 32 + lane].x; };
                            if (count & 1) g1_madd(acc, load_buf(count - 1));
                            affine_round(pairs, lane, load_buf, load_buf_x, prefix, dst);
                        }
                        cur = dst;
                        count = pairs;
                        level++;
                    }
                    // 3. the rest in XYZZ coordinates
#pragma unroll 1
                    for (uint32_t j = 0; j < count; j++) g1_madd(acc, level == 0 ? load_ref(j) : cur[(size_t)j * 32 + lane]);
                }
                sm[t] = acc;
            }
            DR_BLOCK_SYNC();
            for (uint32_t stride = 16; stride > 0; stride >>= 1) {  // fold the 32 lanes of every warp
                DR_THREAD_LOOP(t, ctx) {
                    if ((t % 32) < stride) {
                        G1 a = sm[t];
                        g1_add(a, sm[t + stride]);
                        sm[t] = a;
                    }
                }
                DR_BLOCK_SYNC();
            }
            DR_THREAD_LOOP(t, ctx) {
                const uint32_t item = it * total_slots + ctx.bx * warps + t / 32;
                if ((t % 32) == 0 && item < items) partials[item] = sm[t];
            }
            DR_BLOCK_SYNC();
        }
    }
};

// Sum `slices` partials per MSM and normalise to affine.  `lanes` (a power of two dividing the block size, <= 32) threads per
// MSM: each folds a strided share of the slices, a shared-memory tree folds the lanes.  Small batches are cut into many slices
// to fill the machine, and a serial fold of those was most of a single proof's latency.
DR_HD uint32_t commit_finish_lanes(uint32_t slices) {
    uint32_t l = 1;
    while (l < slices && l < 32) l <<= 1;
    return l;
}
struct CommitFinishBody {
    DR_HD void operator()(const BlockCtx& ctx, const G1* partials, uint32_t slices, uint32_t batch, G1Affine* out, uint32_t lanes) const {
        G1* sm = (G1*)ctx.smem;  // nthreads entries when lanes > 1
        const uint32_t per_block = ctx.nthreads / lanes;
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t m = ctx.bx * per_block + t / lanes, lane = t % lanes;
            G1 acc = G1::inf();
            if (m < batch) {
#pragma unroll 1
                for (uint32_t s = lane; s < slices; s += lanes) g1_add(acc, partials[(size_t)m * slices + s]);
                if (lanes == 1) out[m] = g1_to_affine(acc);
            }
            if (lanes > 1) sm[t] = acc;
        }
        if (lanes == 1) return;
        DR_BLOCK_SYNC();
        for (uint32_t stride = lanes >> 1; stride > 0; stride >>= 1) {
            DR_THREAD_LOOP(t, ctx) {
                if ((t % lanes) < stride) {
                    G1 a = sm[t];
                    g1_add(a, sm[t + stride]);
                    sm[t] = a;
                }
            }
            DR_BLOCK_SYNC();
        }
        DR_THREAD_LOOP(t, ctx) {
            const uint32_t m = ctx.bx * per_block + t / lanes;
            if ((t % lanes) == 0 && m < batch) out[m] = g1_to_affine(sm[t]);
        }
    }
};
inline void launch_commit_finish(Stream st, const G1* partials, uint32_t slices, uint32_t batch, G1Affine* out) {
    const uint32_t lanes = commit_finish_lanes(slices), threads = 64, per_block = threads / lanes;
    launch(st, Dim3((batch + per_block - 1) / per_block), threads, lanes > 1 ? threads * sizeof(G1) : 0, CommitFinishBody(), partials, slices, batch, out, lanes);
}

// affine (Montgomery) -> 96-byte uncompressed and/or 48-byte compressed zcash bytes
struct G1EncodeBody {
    DR_HD void operator()(const BlockCtx& ctx, const G1Affine* in, uint32_t count, uint8_t* out96, uint8_t* out48) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t m = ctx.bx * ctx.nthreads + t;
            if (m < count) {
                G1Affine a = in[m];
                if (out96) g1_serialize(out96 + 96 * (size_t)m, a);
                if (out48) g1_compress(out48 + 48 * (size_t)m, a);
            }
        }
    }
};

// 48-byte compressed / 96-byte uncompressed -> affine Montgomery; ok[m] = 0 on a malformed encoding
struct G1DecodeBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* in, uint32_t len, uint32_t count, G1Affine* out, uint8_t* ok) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t m = ctx.bx * ctx.nthreads + t;
            if (m < count) {
                G1Affine a;
                bool good = g1_decode(a, in + (size_t)len * m, (int)len);
                if (!good) a = G1Affine::inf();
                out[m] = a;
                ok[m] = good ? 1 : 0;
            }
        }
    }
};

}  // namespace dr
