// Variable-base G1 multi-scalar multiplication (bucket method) for arbitrary point sets.
//
// Stands in for blst's `P1_Affines.mult_pippenger(points, scalars)` as the reference calls it through
// `KZG.msm_g1` (dot_ring/ring_proof/pcs/kzg.py:147-149) and in the verifier's lhs / rhs folds (kzg.py:295-296,332-333).
// Commitments over the fixed SRS do not come here (they use the window tables of msm.cuh); this path serves point sets
// that are not known in advance and the 2^11 .. 2^20 sweep over a synthetic SRS.
//
// Pipeline (all on device, no host round trips):
//   digits   signed c-bit digits of every scalar + per-bucket histogram (atomics)
//   scan     exclusive prefix sums of the histogram and of the work units (a unit = at most UNIT points of one bucket, so a
//            skewed scalar distribution -- every scalar equal, 0/1-heavy columns -- cannot serialise on one thread)
//   scatter  counting-sort the (point, sign) references by bucket
//   units    one thread per unit: XYZZ mixed additions of its points
//   buckets  one thread per bucket: fold its units
//   reduce   per window, T_w = sum_k k * S_k by segmented running sums, tree-folded; windows shifted by c*w doublings in parallel
#pragma once
#include "g1.cuh"
#include "msm.cuh"
#include "rt.cuh"

namespace dr {

constexpr uint32_t MSM_UNIT = 16;     // points per work unit (small units keep the lanes of a warp in step)
constexpr uint32_t MSM_SEGMENT = 16;  // buckets per running-sum segment (short serial chains; the segments are tree-folded)

// Scalars are not split by the G1 endomorphism here (the commit tables of msm.cuh are): k1 * P + k2 * phi(P) equals k * P only on G1,
// and these point sets come from callers, where blst's mult_pippenger gives the integer multiple k * P for any curve point.  The
// plain recoding is exact for every point without a per-point subgroup test; against the split it has the same number of bucket
// additions and twice the windows to reduce.
struct MsmGeom {
    uint32_t n, c, W, H;  // n points, H = 2^(c-1) buckets per window
    DR_HD uint32_t buckets() const { return W * H; }
};
constexpr uint32_t MSM_BITS = 256;  // scalars below r < 2^255 + the carry of the signed recoding

// scalars: n x 32-byte little-endian (any value < 2^256, reduced mod r here) -> digits[w * n + i]
struct MsmDigitsBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint8_t* scalars_le32, MsmGeom g, int32_t* digits, uint32_t* count) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < g.n) {
                Fr k = fp_from_le_bytes_mod<Fr>(scalars_le32 + 32 * (size_t)i, 32).from_mont();
                uint32_t carry = 0;
#pragma unroll 1
                for (uint32_t w = 0; w < g.W; w++) {
                    int d = msm_digit(k.v, w, g.c, carry);
                    digits[(size_t)w * g.n + i] = d;
                    if (d) atomic_add_u32(&count[w * g.H + (uint32_t)(d < 0 ? -d : d) - 1], 1u);
                }
            }
        }
    }
};

// Exclusive scans of count[b] (-> offset) and of ceil(count[b] / UNIT) (-> unit_offset) in three coalesced passes:
//   A  each block scans SCAN_TILE consecutive buckets in shared memory (ping-pong Hillis-Steele) and records its two totals
//   B  one block turns the per-block totals into exclusive block bases (and writes the grand total of units)
//   C  every element adds its block base; cursor[b] is reset for the scatter pass
constexpr uint32_t SCAN_TILE = 256;
struct MsmScanTileBody {
    DR_HD void operator()(const BlockCtx& ctx, const uint32_t* count, uint32_t nb, uint32_t* offset, uint32_t* unit_offset, uint32_t* block_tot) const {
        uint32_t* sm = (uint32_t*)ctx.smem;  // 4 * SCAN_TILE: two ping-pong pairs (points, units)
        const uint32_t T = ctx.nthreads;     // == SCAN_TILE
        DR_THREAD_LOOP(t, ctx) {
            uint32_t b = ctx.bx * T + t;
            uint32_t cnt = b < nb ? count[b] : 0;
            sm[t] = cnt;
            sm[2 * T + t] = (cnt + MSM_UNIT - 1) / MSM_UNIT;
        }
        DR_BLOCK_SYNC();
        uint32_t src = 0;
        for (uint32_t d = 1; d < T; d <<= 1) {
            DR_THREAD_LOOP(t, ctx) {
                uint32_t dst = src ^ 1;
                sm[dst * T + t] = sm[src * T + t] + (t >= d ? sm[src * T + t - d] : 0);
                sm[(2 + dst) * T + t] = sm[(2 + src) * T + t] + (t >= d ? sm[(2 + src) * T + t - d] : 0);
            }
            DR_BLOCK_SYNC();
            src ^= 1;
        }
        DR_THREAD_LOOP(t, ctx) {
            uint32_t b = ctx.bx * T + t;
            if (b < nb) {  // inclusive -> exclusive
                offset[b] = t ? sm[src * T + t - 1] : 0;
                unit_offset[b] = t ? sm[(2 + src) * T + t - 1] : 0;
            }
            if (t == T - 1) {
                block_tot[2 * ctx.bx] = sm[src * T + t];
                block_tot[2 * ctx.bx + 1] = sm[(2 + src) * T + t];
            }
        }
    }
};
struct MsmScanBlocksBody {  // one block, one thread per chunk of tiles; nblocks is small (<= 2048)
    DR_HD void operator()(const BlockCtx& ctx, uint32_t* block_tot, uint32_t nblocks, uint32_t* totals) const {
        DR_THREAD_LOOP(t, ctx) {
            if (t == 0) {
                uint32_t a = 0, u = 0;
                for (uint32_t i = 0; i < nblocks; i++) {
                    uint32_t ca = block_tot[2 * i], cu = block_tot[2 * i + 1];
                    block_tot[2 * i] = a;
                    block_tot[2 * i + 1] = u;
                    a += ca;
                    u += cu;
                }
                totals[0] = u;
            }
        }
    }
};
struct MsmScanApplyBody {
    DR_HD void operator()(const BlockCtx& ctx, uint32_t nb, const uint32_t* block_tot, uint32_t* offset, uint32_t* unit_offset, uint32_t* cursor) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t b = ctx.bx * ctx.nthreads + t;
            if (b < nb) {
                offset[b] += block_tot[2 * ctx.bx];
                unit_offset[b] += block_tot[2 * ctx.bx + 1];
                cursor[b] = 0;
            }
        }
    }
};

// refs[offset[b] + slot] = point index | sign << 31
struct MsmScatterBody {
    DR_HD void operator()(const BlockCtx& ctx, MsmGeom g, const int32_t* digits, const uint32_t* offset, uint32_t* cursor, uint32_t* refs) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < g.n) {
#pragma unroll 1
                for (uint32_t w = 0; w < g.W; w++) {
                    int d = digits[(size_t)w * g.n + i];
                    if (d) {
                        uint32_t b = w * g.H + (uint32_t)(d < 0 ? -d : d) - 1;
                        uint32_t slot = atomic_add_u32(&cursor[b], 1u);
                        refs[offset[b] + slot] = i | (d < 0 ? 0x80000000u : 0u);
                    }
                }
            }
        }
    }
};

// unit u belongs to the bucket b with unit_offset[b] <= u < unit_offset[b + 1] (binary search)
struct MsmUnitSumBody {
    DR_HD void operator()(const BlockCtx& ctx, MsmGeom g, const G1Affine* points, const uint32_t* count, const uint32_t* offset, const uint32_t* unit_offset,
                          const uint32_t* totals, const uint32_t* refs, G1* unit_sum) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t u = ctx.bx * ctx.nthreads + t;
            if (u < totals[0]) {
                uint32_t lo = 0, hi = g.buckets() - 1;
                while (lo < hi) {  // last bucket with unit_offset <= u
                    uint32_t mid = (lo + hi + 1) >> 1;
                    if (unit_offset[mid] <= u) lo = mid;
                    else hi = mid - 1;
                }
                // empty buckets share their unit_offset with the next one: step to the owner
                uint32_t b = lo;
                uint32_t first = offset[b] + (u - unit_offset[b]) * MSM_UNIT;
                uint32_t end = offset[b] + count[b];
                uint32_t stop = first + MSM_UNIT < end ? first + MSM_UNIT : end;
                G1 acc = G1::inf();
#pragma unroll 1
                for (uint32_t r = first; r < stop; r++) {
                    uint32_t ref = refs[r];
                    g1_madd(acc, points[ref & 0x7FFFFFFFu], (ref >> 31) != 0);
                }
                unit_sum[u] = acc;
            }
        }
    }
};

// Buckets with few units are folded by one thread; a bucket that received a large share of the points (the top window only
// spans the few leading bits of the scalars, and skewed scalar distributions concentrate everything in a handful of buckets)
// gets a whole CTA: strided partial sums, then a shared-memory tree.
constexpr uint32_t MSM_FOLD_SERIAL = 32;
struct MsmBucketFoldBody {
    DR_HD void operator()(const BlockCtx& ctx, MsmGeom g, const uint32_t* count, const uint32_t* unit_offset, const G1* unit_sum, G1* bucket) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t b = ctx.bx * ctx.nthreads + t;
            if (b < g.buckets()) {
                uint32_t units = (count[b] + MSM_UNIT - 1) / MSM_UNIT;
                if (units <= MSM_FOLD_SERIAL) {
                    G1 acc = G1::inf();
#pragma unroll 1
                    for (uint32_t u = 0; u < units; u++) g1_add(acc, unit_sum[unit_offset[b] + u]);
                    bucket[b] = acc;
                }
            }
        }
    }
};
struct MsmBucketFoldHeavyBody {  // grid = buckets; CTAs of light buckets exit at once
    DR_HD void operator()(const BlockCtx& ctx, const uint32_t* count, const uint32_t* unit_offset, const G1* unit_sum, G1* bucket) const {
        const uint32_t b = ctx.bx;
        const uint32_t units = (count[b] + MSM_UNIT - 1) / MSM_UNIT;
        if (units <= MSM_FOLD_SERIAL) return;
        G1* sm = (G1*)ctx.smem;
        DR_THREAD_LOOP(t, ctx) {
            G1 acc = G1::inf();
#pragma unroll 1
            for (uint32_t u = t; u < units; u += ctx.nthreads) g1_add(acc, unit_sum[unit_offset[b] + u]);
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
            if (t == 0) bucket[b] = sm[0];
        }
    }
};

// segment s of window w covers buckets k = lo..hi (1-based digit values): out = sum_k k * S_k
struct MsmSegmentReduceBody {
    DR_HD void operator()(const BlockCtx& ctx, MsmGeom g, const G1* bucket, uint32_t segs_per_window, G1* seg_sum) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t id = ctx.bx * ctx.nthreads + t;
            if (id < g.W * segs_per_window) {
                uint32_t w = id / segs_per_window, s = id % segs_per_window;
                uint32_t lo = s * MSM_SEGMENT + 1;
                uint32_t hi = lo + MSM_SEGMENT - 1 < g.H ? lo + MSM_SEGMENT - 1 : g.H;
                G1 running = G1::inf(), acc = G1::inf();
#pragma unroll 1
                for (uint32_t k = hi; k >= lo; k--) {
                    g1_add(running, bucket[(size_t)w * g.H + k - 1]);
                    g1_add(acc, running);  // after the loop: sum (k - lo + 1) * S_k
                }
                // + (lo - 1) * sum S_k
                uint32_t m = lo - 1;
                if (m) {
                    G1 add = G1::inf();
#pragma unroll 1
                    for (int bit = 31; bit >= 0; bit--) {
                        if (!add.is_inf()) add = g1_dbl(add);
                        if ((m >> bit) & 1) g1_add(add, running);
                    }
                    g1_add(acc, add);
                }
                seg_sum[id] = acc;
            }
        }
    }
};

// block w: tree-fold the window's segments -> T_w
struct MsmWindowFoldBody {
    DR_HD void operator()(const BlockCtx& ctx, const G1* seg_sum, uint32_t segs_per_window, G1* window_sum) const {
        G1* sm = (G1*)ctx.smem;
        DR_THREAD_LOOP(t, ctx) {
            G1 acc = G1::inf();
#pragma unroll 1
            for (uint32_t s = t; s < segs_per_window; s += ctx.nthreads) g1_add(acc, seg_sum[(size_t)ctx.bx * segs_per_window + s]);
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
            if (t == 0) window_sum[ctx.bx] = sm[0];
        }
    }
};
// sum_w 2^(c w) T_w: thread w shifts its window by c*w doublings, then a tree adds the W shifted sums
struct MsmFinalBody {
    DR_HD void operator()(const BlockCtx& ctx, MsmGeom g, const G1* window_sum, G1Affine* out) const {
        G1* sm = (G1*)ctx.smem;  // nthreads entries (power of two >= W)
        DR_THREAD_LOOP(t, ctx) {
            G1 acc = G1::inf();
            if (t < g.W) {
                acc = window_sum[t];
#pragma unroll 1
                for (uint32_t k = 0; k < g.c * t; k++) acc = g1_dbl(acc);
            }
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
            if (t == 0) *out = g1_to_affine(sm[0]);
        }
    }
};

// ---- synthetic SRS for the sweep: P_i = tau^i * G ----------------------------------------------------------------
struct SyntheticSrsBody {  // out[i] = tau^(offset + i) * G
    DR_HD void operator()(const BlockCtx& ctx, G1Affine gen, Fr tau, uint32_t offset, uint32_t n, G1Affine* out) const {
        DR_THREAD_LOOP(t, ctx) {
            uint32_t i = ctx.bx * ctx.nthreads + t;
            if (i < n) {
                Fr e = Fr::one(), base = tau;
                uint32_t k = offset + i;
#pragma unroll 1
                while (k) {
                    if (k & 1) e = e * base;
                    base = base.sqr();
                    k >>= 1;
                }
                Fr raw = e.from_mont();
                out[i] = g1_to_affine(g1_mul_limbs(G1::from_affine(gen), raw.v));
            }
        }
    }
};

}  // namespace dr
