// Warp-cooperative reservoir statistics (one warp per reservoir).
//
// Computes the five features of ReservoirSampler.get_features
// (reference: simulation-mode/problem-01-reservoir-sampling/src/reservoir.py:105-196)
//   mean, p90 (numpy 'linear' percentile), std (ddof 0),
//   mean_decay = sum(v*w)/sum(w), p90_decay = weighted percentile,
//   with w = decay^(now - timestamp).
//
// Layout: the K<=128 slots of one reservoir are spread over the 32 lanes,
// EPL = 1, 2 or 4 consecutive slots per lane (one 32/64/128-bit load each).
//
// Order statistics come from a per-slot RANK (position of the slot's value in
// ascending order).  Ranks are either computed from scratch -- an in-register
// bitonic network over (value, slot) pairs, intra-lane stages as compare-
// exchanges and inter-lane stages as shuffles -- or, when the caller keeps the
// ranks of the previous step, updated incrementally for the few slots that
// Algorithm R replaced (remove the old rank, count-and-insert the new value:
// ~50 instructions per replaced slot instead of a ~600-instruction sort).
// Values and weights are then scattered by rank into a 1 KB per-warp shared-
// memory scratch, which makes "value at rank r" a broadcast read and the
// weighted percentile a blocked read + warp scan.
//
// The decay weights only matter up to a common factor (both weighted outputs
// are ratios / order decisions), so the fast path evaluates them in float32
// relative to the newest timestamp, w = 2^(log2(decay) * (t_max - t)), and
// takes the weighted percentile index from a float32 warp scan.  If any
// cumulative weight lies within a relative margin of the 0.9*W cutoff the
// warp (uniformly) re-does the decision the way the reference does it:
// float64 pow(decay, now - t) and a strictly sequential float64 cumsum in
// value order (np.cumsum + np.searchsorted, reservoir.py:186-190).
#pragma once
#include "mlb_common.cuh"

namespace mlb {

// relative distance to the cutoff below which the float32 index decision is
// not trusted (error bound of the fast path is < 1e-5 * W, see DESIGN.md)
#define MLB_WP_MARGIN 5e-5f

// One compare-exchange stage of the bitonic network; SIZE / STRIDE are template
// constants so every register index is static (no local-memory arrays).
template <int EPL, int SIZE, int STRIDE>
__device__ __forceinline__ void bitonic_stage(float (&k)[EPL], float (&p)[EPL], int lane) {
    // Branch-free compare-exchange: the new key is min or max (FMNMX + FSEL); the payload
    // follows iff the key changed, so equal keys keep their own payload on both sides.
    if constexpr (STRIDE >= EPL) {
        constexpr int LSTRIDE = STRIDE / EPL;
        const bool keep_min = (((lane * EPL) & SIZE) == 0) == ((lane & LSTRIDE) == 0);
#pragma unroll
        for (int r = 0; r < EPL; r++) {
            const float ok = __shfl_xor_sync(MLB_FULL, k[r], LSTRIDE);
            const float op = __shfl_xor_sync(MLB_FULL, p[r], LSTRIDE);
            const float nk = keep_min ? fminf(k[r], ok) : fmaxf(k[r], ok);
            p[r] = (nk != k[r]) ? op : p[r];
            k[r] = nk;
        }
    } else {
#pragma unroll
        for (int r = 0; r < EPL; r++) {
            if ((r & STRIDE) == 0) {
                const int r2 = r | STRIDE;
                const bool up = (((lane * EPL + r) & SIZE) == 0);
                const float a = k[r], b = k[r2], pa = p[r], pb = p[r2];
                const float lo = fminf(a, b), hi = fmaxf(a, b);
                const float na = up ? lo : hi;
                const bool sw = na != a;
                k[r] = na;
                k[r2] = up ? hi : lo;
                p[r] = sw ? pb : pa;
                p[r2] = sw ? pa : pb;
            }
        }
    }
    if constexpr (STRIDE > 1) bitonic_stage<EPL, SIZE, STRIDE / 2>(k, p, lane);
}

template <int EPL, int SIZE>
__device__ __forceinline__ void bitonic_merge_levels(float (&k)[EPL], float (&p)[EPL], int lane) {
    bitonic_stage<EPL, SIZE, SIZE / 2>(k, p, lane);
    if constexpr (SIZE < 32 * EPL) bitonic_merge_levels<EPL, SIZE * 2>(k, p, lane);
}

// ascending sort of the 32*EPL (key, payload) pairs, element index = lane*EPL + r
template <int EPL>
__device__ __forceinline__ void bitonic_sort_kv(float (&k)[EPL], float (&p)[EPL], int lane) {
    bitonic_merge_levels<EPL, 2>(k, p, lane);
}

template <int EPL>
__device__ __forceinline__ void load_slots(const float* __restrict__ base, int lane, float (&x)[EPL]) {
    if constexpr (EPL == 4) {
        const float4 q = ldg_stream4(base + lane * 4);
        x[0] = q.x; x[1] = q.y; x[2] = q.z; x[3] = q.w;
    } else if constexpr (EPL == 2) {
        const float2 q = ldg_stream2(base + lane * 2);
        x[0] = q.x; x[1] = q.y;
    } else {
        x[0] = ldg_stream1(base + lane);
    }
}

// ranks are one byte per slot in global memory
template <int EPL>
__device__ __forceinline__ void load_ranks(const uint8_t* __restrict__ base, int lane, int (&rk)[EPL]) {
    if constexpr (EPL == 4) {
        const uint32_t q = *reinterpret_cast<const uint32_t*>(base + lane * 4);
        rk[0] = q & 255; rk[1] = (q >> 8) & 255; rk[2] = (q >> 16) & 255; rk[3] = q >> 24;
    } else if constexpr (EPL == 2) {
        const uint32_t q = *reinterpret_cast<const uint16_t*>(base + lane * 2);
        rk[0] = q & 255; rk[1] = q >> 8;
    } else {
        rk[0] = base[lane];
    }
}
template <int EPL>
__device__ __forceinline__ void store_ranks(uint8_t* __restrict__ base, int lane, const int (&rk)[EPL]) {
    if constexpr (EPL == 4) {
        *reinterpret_cast<uint32_t*>(base + lane * 4) =
            (uint32_t)(rk[0] & 255) | ((uint32_t)(rk[1] & 255) << 8) | ((uint32_t)(rk[2] & 255) << 16) | ((uint32_t)rk[3] << 24);
    } else if constexpr (EPL == 2) {
        *reinterpret_cast<uint16_t*>(base + lane * 2) = (uint16_t)((rk[0] & 255) | ((rk[1] & 255) << 8));
    } else {
        base[lane] = (uint8_t)rk[0];
    }
}

// per-warp shared-memory scratch: 128 (value, weight) pairs in rank order
struct WarpScratch {
    float2* vw;
};
#define MLB_SCRATCH_BYTES 1024

// Ranks from scratch: bitonic sort of (value, slot) pairs, then transpose position->slot
// into slot->position through shared-memory bytes.  Slots >= n get rank 255.
// noinline: cold once reservoirs are full and ranks are maintained incrementally; keeping
// it out of line keeps the steady-state loop inside the instruction cache.  Values go in by
// value and the EPL ranks come back packed in one word so that nothing lives in local memory.
template <int EPL>
struct SlotVals {
    float x[EPL];
};

template <int EPL>
__device__ __noinline__ uint32_t ranks_full_sort_packed(SlotVals<EPL> v, int n, float2* scratch) {
    const int lane = lane_id();
    float k[EPL], p[EPL];
#pragma unroll
    for (int r = 0; r < EPL; r++) {
        const int slot = lane * EPL + r;
        k[r] = slot < n ? v.x[r] : MLB_INF;  // padding sorts to the end
        p[r] = __int_as_float(slot);
    }
    bitonic_sort_kv<EPL>(k, p, lane);
    uint8_t* sb = reinterpret_cast<uint8_t*>(scratch);
#pragma unroll
    for (int r = 0; r < EPL; r++) {
        const int pos = lane * EPL + r;
        sb[__float_as_int(p[r])] = (uint8_t)(pos < n ? pos : 255);
    }
    __syncwarp();
    uint32_t packed = 0;
#pragma unroll
    for (int r = 0; r < EPL; r++) packed |= (uint32_t)sb[lane * EPL + r] << (8 * r);
    __syncwarp();
    return packed;
}

template <int EPL>
__device__ __forceinline__ void ranks_full_sort(const float (&v)[EPL], int n, int (&rk)[EPL],
                                                const WarpScratch& sc) {
    SlotVals<EPL> sv;
#pragma unroll
    for (int r = 0; r < EPL; r++) sv.x[r] = v[r];
    const uint32_t packed = ranks_full_sort_packed<EPL>(sv, n, sc.vw);
#pragma unroll
    for (int r = 0; r < EPL; r++) rk[r] = (packed >> (8 * r)) & 255u;
}

// Cold paths of the weighted percentile, taken when the float32 cumulative weights come
// within MLB_WP_MARGIN of the cutoff.  st[p].y = timestamp of the element at rank p, n <= 128.
//
// Tier 2: float64 weights 2^(log2(decay) * (tmax - t)) and a float64 warp scan; decides unless
// a cumulative weight is within 1e-9 (relative) of the cutoff, i.e. a genuine tie.
static __device__ __noinline__ int weighted_index_scan_f64(const float2* st, int n, float tmax, double decay,
                                                           bool* ambiguous) {
    const int lane = lane_id();
    const double l2d = log2(decay);
    double w[4], c[4];
    double carry = 0.0;
#pragma unroll
    for (int k = 0; k < 4; k++) {  // position p = k*32 + lane
        const int pos = k * 32 + lane;
        w[k] = pos < n ? exp2(l2d * ((double)tmax - (double)st[pos].y)) : 0.0;
        double sc = w[k];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double y = __shfl_up_sync(MLB_FULL, sc, o);
            if (lane >= o) sc += y;
        }
        c[k] = carry + sc;
        carry = __shfl_sync(MLB_FULL, c[k], 31);
    }
    const double cut = 0.9 * carry;
    int below = 0;
    double dmin = 1.0e308;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const bool valid = k * 32 + lane < n;
        below += (valid && c[k] < cut) ? 1 : 0;
        dmin = valid ? fmin(dmin, fabs(c[k] - cut)) : dmin;
    }
    dmin = warp_min(dmin);
    *ambiguous = dmin < 1e-9 * carry;
    return __reduce_add_sync(MLB_FULL, below);
}

// Correctly rounded decay^y for tier 3.  Tier 3 runs when a cumulative weight sits within 1e-9 of the cutoff,
// in practice an exact tie in real arithmetic (e.g. ten samples of one timestamp, the cutoff on the ninth).  There
// the reference's decision hangs on the last bit of each weight, which the host's pow rounds correctly for all but a
// few arguments while CUDA's pow may be 2 ulp off.  exp(y * ln(decay)) in double-double arithmetic (~2^-95 relative
// error) rounds correctly.
// Explicitly rounded operations: a contraction into fma would break the error-free transforms.
struct DD {
    double hi, lo;
};
__device__ __forceinline__ double dd_rn_add(double a, double b) {
    return __dadd_rn(a, b);
}
__device__ __forceinline__ double dd_rn_mul(double a, double b) {
    return __dmul_rn(a, b);
}
__device__ __forceinline__ double dd_rn_fma(double a, double b, double c) {
    return __fma_rn(a, b, c);
}
__device__ __forceinline__ DD dd_two_sum(double a, double b) {
    const double s = dd_rn_add(a, b), bb = dd_rn_add(s, -a);
    return {s, dd_rn_add(dd_rn_add(a, -dd_rn_add(s, -bb)), dd_rn_add(b, -bb))};
}
__device__ __forceinline__ DD dd_quick_two_sum(double a, double b) {   // |a| >= |b|
    const double s = dd_rn_add(a, b);
    return {s, dd_rn_add(b, -dd_rn_add(s, -a))};
}
__device__ __forceinline__ DD dd_add(DD a, DD b) {
    DD s = dd_two_sum(a.hi, b.hi);
    const DD t = dd_two_sum(a.lo, b.lo);
    s = dd_quick_two_sum(s.hi, dd_rn_add(s.lo, t.hi));
    return dd_quick_two_sum(s.hi, dd_rn_add(s.lo, t.lo));
}
__device__ __forceinline__ DD dd_mul(DD a, DD b) {
    const double p = dd_rn_mul(a.hi, b.hi);
    const double e = dd_rn_fma(a.lo, b.hi, dd_rn_fma(a.hi, b.lo, dd_rn_fma(a.hi, b.hi, -p)));
    return dd_quick_two_sum(p, e);
}
__device__ __forceinline__ DD dd_mul_d(DD a, double b) {
    const double p = dd_rn_mul(a.hi, b);
    return dd_quick_two_sum(p, dd_rn_fma(a.lo, b, dd_rn_fma(a.hi, b, -p)));
}
// e^z = 2^k e^r, e^r = (e^(r/1024))^1024: Taylor series of e^s - 1 to s^9 (|s| < 3.4e-4), then ten squarings of
// 1 + x as x <- 2x + x^2.  Returns the double-double value, |z| < 700.
__device__ inline DD dd_exp(DD z) {
    const DD ln2 = {0x1.62e42fefa39efp-1, 0x1.abc9e3b39803fp-56};
    const double k = rint(dd_rn_mul(z.hi, 0x1.71547652b82fep0));
    DD r = dd_add(z, dd_mul_d(ln2, -k));
    r.hi = dd_rn_mul(r.hi, 0x1p-10);
    r.lo = dd_rn_mul(r.lo, 0x1p-10);
    DD p = {0.0, 0.0};
    double fact = 362880.0;                       // 9!
    for (int m = 9; m >= 1; m--) {                // p <- p * s + 1/m!
        const double c = 1.0 / fact;
        p = dd_add(dd_mul(p, r), DD{c, dd_rn_fma(-c, fact, 1.0) / fact});
        fact /= m;
    }
    DD x = dd_mul(p, r);
    for (int i = 0; i < 10; i++) x = dd_add(DD{dd_rn_mul(x.hi, 2.0), dd_rn_mul(x.lo, 2.0)}, dd_mul(x, x));
    const DD e = dd_add(DD{1.0, 0.0}, x);
    return {ldexp(e.hi, (int)k), ldexp(e.lo, (int)k)};
}
// ln(decay) as a double-double: one Newton step on log(decay).
__device__ inline DD dd_log(double d) {
    const double l0 = log(d);
    const DD e = dd_exp(DD{l0, 0.0});
    const DD num = dd_add(DD{d, 0.0}, DD{-e.hi, -e.lo});
    return dd_two_sum(l0, dd_rn_add(num.hi, num.lo) / e.hi);
}
// decay^y rounded to nearest, given ln_decay = dd_log(decay).
__device__ inline double pow_cr(double decay, DD ln_decay, double y) {
    if (y == 0.0 || decay == 1.0) return 1.0;
    const DD z = dd_mul_d(ln_decay, y);
    // beyond e^-700 (a weight older than ~6600 s at decay 0.9) the result leaves the normal range, where ldexp would
    // round a second time: CUDA's pow decides there, so a tie among weights that small may go the other way
    if (!(fabs(z.hi) < 700.0)) return pow(decay, y);
    return dd_exp(z).hi;
}

// Tier 3: the reference's own arithmetic (reservoir.py:148-149,181-196): w = pow(decay, now - t)
// (correctly rounded, as the host's pow) and a strictly sequential cumsum in value order.  Returns the
// searchsorted-left index of 0.9 * cumsum[-1] (n if none).
static __device__ __noinline__ int weighted_index_f64(const float2* st, int n, float now, double decay) {
    const int lane = lane_id();
    const DD ln_decay = dd_log(decay);
    double w[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int pos = k * 32 + lane;
        w[k] = pos < n ? pow_cr(decay, ln_decay, (double)now - (double)st[pos].y) : 0.0;
    }
    double c = 0.0;
#pragma unroll 1
    for (int p = 0; p < n; p++) {
        const int k = p >> 5;
        const double wk = k == 0 ? w[0] : (k == 1 ? w[1] : (k == 2 ? w[2] : w[3]));
        c += __shfl_sync(MLB_FULL, wk, p & 31);
    }
    const double cut = 0.9 * c;  // percentile * cumsum[-1]
    c = 0.0;
    int idx = n;
#pragma unroll 1
    for (int p = 0; p < n; p++) {
        const int k = p >> 5;
        const double wk = k == 0 ? w[0] : (k == 1 ? w[1] : (k == 2 ? w[2] : w[3]));
        c += __shfl_sync(MLB_FULL, wk, p & 31);
        if (c >= cut) {
            idx = p;
            break;
        }
    }
    return idx;
}

// Both float64 tiers; out of line so the steady-state loop stays small.  Returns the index, plus 0x100 when tier 2
// found an exact tie and tier 3 decided it.
template <int EPL>
__device__ __noinline__ int weighted_index_exact(SlotVals<EPL> t, uint32_t rk_packed, int n, float tmax, float now,
                                                 double decay, float2* vw) {
    const int s0 = lane_id() * EPL;
    __syncwarp();
#pragma unroll
    for (int r = 0; r < EPL; r++)
        if (s0 + r < n) vw[(rk_packed >> (8 * r)) & 255u].y = t.x[r];  // weights are no longer needed
    __syncwarp();
    bool ambiguous;
    int idx = weighted_index_scan_f64(vw, n, tmax, decay, &ambiguous);
    if (ambiguous) idx = weighted_index_f64(vw, n, now, decay) | 0x100;
    return idx;
}

__device__ __forceinline__ float fast_rcp(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float fast_sqrt(float x) {
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// The five features given slot-ordered values/timestamps and valid ranks.
// FULL: all 32*EPL slots are valid (n == 32*EPL), which makes n and everything derived from
// it (p90 positions, interpolation weight, 1/n) compile-time constants.  `tie` is set when the
// p90_decay index sits on an exact tie (decided by tier 3).
template <int EPL, bool FULL>
__device__ __forceinline__ void features_ranked(const float (&v)[EPL], const float (&t)[EPL],
                                                const int (&rk)[EPL], int n_, float now, double decay,
                                                float log2_decay, const WarpScratch& sc, float (&out)[5],
                                                bool& tie) {
    const int lane = lane_id();
    const int s0 = lane * EPL;
    const int n = FULL ? 32 * EPL : n_;
    tie = false;
    // ---- mean (np.mean on float32: reservoir.py:143), newest timestamp
    float s = 0.f, tmax = -MLB_INF;
#pragma unroll
    for (int r = 0; r < EPL; r++) {
        const bool valid = FULL || s0 + r < n;
        s += valid ? v[r] : 0.f;
        tmax = valid ? fmaxf(tmax, t[r]) : tmax;
    }
    const float nf = (float)n;
    const float mean = warp_sum(s) / nf;
    tmax = f32_from_orderable(__reduce_max_sync(MLB_FULL, f32_orderable(tmax)));
    // ---- std (np.std, two passes: reservoir.py:145); decay weights relative to the newest
    //      sample (float32 fast path); (value, weight) scattered by rank
    float s2 = 0.f, svw = 0.f;
#pragma unroll
    for (int r = 0; r < EPL; r++) {
        const bool valid = FULL || s0 + r < n;
        const float d = v[r] - mean;
        s2 += valid ? d * d : 0.f;
        const float w = valid ? fast_exp2(log2_decay * (tmax - t[r])) : 0.f;
        svw += valid ? v[r] * w : 0.f;
        const int pos = valid ? rk[r] : s0 + r;  // ranks cover [0,n); slots >= n pad positions >= n
        sc.vw[pos] = make_float2(v[r], w);
    }
    const float sd = fast_sqrt(warp_sum(s2) / nf);
    svw = warp_sum(svw);
    __syncwarp();
    // ---- weighted percentile: blocked read of weights in rank order + warp scan
    float cum[EPL];
    float sw = 0.f;
#pragma unroll
    for (int r = 0; r < EPL; r += 2) {
        if constexpr (EPL == 1) {
            sw += sc.vw[s0].y;
            cum[0] = sw;
        } else {
            const float4 q = *reinterpret_cast<const float4*>(sc.vw + s0 + r);
            sw += q.y;
            cum[r] = sw;
            sw += q.w;
            cum[r + 1] = sw;
        }
    }
    const float incl = warp_scan_incl(sw, lane);
    const float W = __shfl_sync(MLB_FULL, incl, 31);
    const float mean_decay = svw * fast_rcp(W);
    const float rel = 0.9f * W - (incl - sw);  // cutoff relative to this lane's first position
    int below = 0;
    float dmin = MLB_INF;
#pragma unroll
    for (int r = 0; r < EPL; r++) {
        const bool valid = FULL || s0 + r < n;  // here s0+r is a POSITION in rank order
        below += (valid && cum[r] < rel) ? 1 : 0;
        dmin = valid ? fminf(dmin, fabsf(cum[r] - rel)) : dmin;
    }
    int idx = __reduce_add_sync(MLB_FULL, below);
    const uint32_t dmin_bits = __reduce_min_sync(MLB_FULL, __float_as_uint(dmin));
    if (__uint_as_float(dmin_bits) < MLB_WP_MARGIN * W) {
        // ---- not trusted: redo the decision in the reference's float64 arithmetic
        SlotVals<EPL> tv;
        uint32_t packed = 0;
#pragma unroll
        for (int r = 0; r < EPL; r++) {
            tv.x[r] = t[r];
            packed |= (uint32_t)(rk[r] & 255) << (8 * r);
        }
        idx = weighted_index_exact<EPL>(tv, packed, n, tmax, now, decay, sc.vw);
        tie = idx >= 0x100;
        idx &= 0xff;
    }
    idx = idx > n - 1 ? n - 1 : idx;  // reservoir.py:193-194
    // ---- p90 = np.percentile(values, 90): float32 'linear' rule of numpy >= 2
    const float vidx = (float)(n - 1) * (90.0f / 100.0f);
    const float fl = floorf(vidx);
    int lo = (int)fl, hi = lo + 1;
    if (vidx >= (float)(n - 1)) { lo = n - 1; hi = n - 1; }
    hi = hi > n - 1 ? n - 1 : hi;
    const float gamma = vidx - fl;
    const float a = sc.vw[lo].x, b = sc.vw[hi].x;
    const float p90_decay = sc.vw[idx].x;
    const float diff = __fsub_rn(b, a);
    float p90 = __fadd_rn(a, __fmul_rn(diff, gamma));
    if (gamma >= 0.5f) p90 = __fsub_rn(b, __fmul_rn(diff, __fsub_rn(1.0f, gamma)));
    __syncwarp();  // scratch is reused by the next reservoir
    out[0] = mean;
    out[1] = p90;
    out[2] = sd;
    out[3] = mean_decay;
    out[4] = p90_decay;
}

// Ranks from scratch, then the features: the stateless form (reservoir_features_kernel) and
// every case of the env step that is not "full reservoir, a few replaced slots".  `ranks`
// (may be null) receives the ranks for later incremental updates.  n = min(count, K) >= 1.
template <int EPL>
__device__ __forceinline__ void features_sorted_epl(const float* __restrict__ vals, const float* __restrict__ tss,
                                                    uint8_t* __restrict__ ranks, int n, float now, double decay,
                                                    float log2_decay, const WarpScratch& sc, float (&out)[5],
                                                    bool& tie) {
    const int lane = lane_id();
    float v[EPL], t[EPL];
    int rk[EPL];
    load_slots<EPL>(vals, lane, v);
    load_slots<EPL>(tss, lane, t);
    ranks_full_sort<EPL>(v, n, rk, sc);
    if (ranks) store_ranks<EPL>(ranks, lane, rk);
    if (n == 32 * EPL)
        features_ranked<EPL, true>(v, t, rk, n, now, decay, log2_decay, sc, out, tie);
    else
        features_ranked<EPL, false>(v, t, rk, n, now, decay, log2_decay, sc, out, tie);
}

// ---------------------------------------------------------------------------
// Half-warp forms for the steady state (FULL 128-slot reservoir, ONE replaced slot): the reservoir
// lies on 16 lanes x 8 consecutive slots, so every warp instruction serves TWO reservoirs (one per
// half-warp).  All warp-uniform work -- list decoding, addresses, reductions, scans, broadcasts -- is
// thereby halved per reservoir; the per-element work is unchanged.  hl = lane & 15, half = lane >> 4.
// Every collective keeps the FULL member mask so that the warp stays converged (half masks would let the
// two halves drift apart and be issued separately): shuffles are segmented by width 16, integer REDUX sums
// carry the two halves in separate 16-bit fields, REDUX min / max run once per half with the identity
// contributed by the other half.
__device__ __forceinline__ float half_sum(float v) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(MLB_FULL, v, o, 16);
    return v;
}
__device__ __forceinline__ uint32_t half_reduce_add_u16(uint32_t x, int half) {   // x < 2^16 / 16 per lane
    const uint32_t both = __reduce_add_sync(MLB_FULL, half ? (x << 16) : x);
    return half ? (both >> 16) : (both & 0xffffu);
}
__device__ __forceinline__ uint32_t half_reduce_max(uint32_t x, int half) {
    const uint32_t m0 = __reduce_max_sync(MLB_FULL, half ? 0u : x);
    const uint32_t m1 = __reduce_max_sync(MLB_FULL, half ? x : 0u);
    return half ? m1 : m0;
}
__device__ __forceinline__ uint32_t half_reduce_min(uint32_t x, int half) {
    const uint32_t m0 = __reduce_min_sync(MLB_FULL, half ? 0xffffffffu : x);
    const uint32_t m1 = __reduce_min_sync(MLB_FULL, half ? x : 0xffffffffu);
    return half ? m1 : m0;
}

template <typename T>
__device__ __forceinline__ T pick8(const T (&x)[8], int sub) {
    const T a = (sub & 1) ? x[1] : x[0], b = (sub & 1) ? x[3] : x[2];
    const T c = (sub & 1) ? x[5] : x[4], d = (sub & 1) ? x[7] : x[6];
    const T lo = (sub & 2) ? b : a, hi = (sub & 2) ? d : c;
    return (sub & 4) ? hi : lo;
}

// Incremental rank maintenance for a reservoir in which Algorithm R replaced a few slots
// (rank_replace_one_h16, rank_update_h16).  v[] already holds the new values, rkp[] the ranks of
// the previous contents.  Any order of equal values is a valid sorted order, and the stored
// ranks may hold tied values in ANY order (the bitonic sort does not order ties), so the
// update must not assume one: a new value is inserted AFTER every present element that
// equals it -- "before" = (v_i <= x), "after" = (v_i > x), which is consistent with whatever
// order the ties already have.  (Ranking ties by slot index instead, as this code first did,
// produced duplicate ranks when a third equal value met a tied pair that a re-sort had left in
// non-slot order; float32 durations taken as differences of timestamps are quantised, so such
// triple ties do occur at scale: tools/determinism_probe.py, tests/test_gpu_ties.py.)
//
// One replaced slot c of a FULL reservoir (the common case), ranks packed one per byte in two words: take out c's old
// rank, count the elements below the new value x and shift the others with SWAR arithmetic.  v_i <= x is tested as
// v_i < nextup(x) for every slot but c itself (which holds x and must not count); ranks above the removed one move
// down (bytes <= 127, so the borrow never crosses a byte), ranks at or above the inserted one move up.
__device__ __forceinline__ void rank_replace_one_h16(const float (&v)[8], uint32_t (&rkp)[2], int c, int hl,
                                                     int half) {
    const int sub = c & 7, lc = c >> 3;
    const float x = __shfl_sync(MLB_FULL, pick8(v, sub), lc, 16) + 0.0f;   // -0 -> +0
    const uint32_t wsel = (sub & 4) ? rkp[1] : rkp[0];
    const uint32_t r_old = (__shfl_sync(MLB_FULL, wsel, lc, 16) >> (8 * (sub & 3))) & 255u;
    const uint32_t xb = __float_as_uint(x);
    const float xup = __uint_as_float((xb >> 31) ? xb - 1u : xb + 1u);
    const int dl = c - hl * 8;  // slot r == dl of this lane is c (it holds x itself and must not count)
    uint32_t bef0 = 0, bef1 = 0;
#pragma unroll
    for (int r = 0; r < 4; r++) {
        bef0 |= v[r] < (r == dl ? x : xup) ? (1u << (8 * r)) : 0u;
        bef1 |= v[r + 4] < (r + 4 == dl ? x : xup) ? (1u << (8 * r)) : 0u;
    }
    const uint32_t r_new = half_reduce_add_u16((uint32_t)(__popc(bef0) + __popc(bef1)), half);
    const uint32_t rep = (r_old + 1u) * 0x01010101u;
    rkp[0] = rkp[0] - ((((rkp[0] | 0x80808080u) - rep) >> 7) & 0x01010101u) + (bef0 ^ 0x01010101u);
    rkp[1] = rkp[1] - ((((rkp[1] | 0x80808080u) - rep) >> 7) & 0x01010101u) + (bef1 ^ 0x01010101u);
    if (hl == lc) {
        const int sh = 8 * (sub & 3);
        if (sub & 4) rkp[1] = (rkp[1] & ~(255u << sh)) | (r_new << sh);
        else rkp[0] = (rkp[0] & ~(255u << sh)) | (r_new << sh);
    }
}

// features_ranked<4, true> on 8 slots per lane; vw = this half's 128-entry scratch.
// Returns false when the float32 weighted-percentile decision is not trusted (the caller hands the reservoir to
// warp_features_ranked_exact) instead of calling the float64 tiers, so that the hot loop contains no calls.
__device__ __forceinline__ bool features_full_h16(const float (&v)[8], const float (&t)[8], const uint32_t (&rkp)[2],
                                                  float log2_decay, float2* vw, int hl, int half,
                                                  float (&out)[5]) {
    const float s = ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
    const float tm = fmaxf(fmaxf(fmaxf(t[0], t[1]), fmaxf(t[2], t[3])), fmaxf(fmaxf(t[4], t[5]), fmaxf(t[6], t[7])));
    const float mean = half_sum(s) * (1.0f / 128.0f);
    const float tmax = f32_from_orderable(half_reduce_max(f32_orderable(tm), half));
    float s2 = 0.f, svw = 0.f;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const float dv = v[r] - mean;
        s2 += dv * dv;
        const float w = fast_exp2(log2_decay * (tmax - t[r]));
        svw += v[r] * w;
        // rank p lives at index (p & 7) * 16 + (p >> 3): lane hl then reads its eight consecutive ranks
        // 8 * hl + r at index r * 16 + hl -- consecutive lanes, consecutive words, no bank conflicts
        const uint32_t pos = (rkp[r >> 2] >> (8 * (r & 3))) & 255u;
        vw[((pos & 7u) << 4) | (pos >> 3)] = make_float2(v[r], w);
    }
    const float sd = fast_sqrt(half_sum(s2) * (1.0f / 128.0f));
    svw = half_sum(svw);
    __syncwarp();
    float cum[8];
    float sw = 0.f;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        sw += vw[r * 16 + hl].y;
        cum[r] = sw;
    }
    float incl = sw;
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) {
        const float y = __shfl_up_sync(MLB_FULL, incl, o, 16);
        if (hl >= o) incl += y;
    }
    const float W = __shfl_sync(MLB_FULL, incl, 15, 16);
    const float mean_decay = svw * fast_rcp(W);
    const float rel = 0.9f * W - (incl - sw);
    int below = 0;
    float dmin = MLB_INF;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        below += cum[r] < rel ? 1 : 0;
        dmin = fminf(dmin, fabsf(cum[r] - rel));
    }
    int idx = (int)half_reduce_add_u16((uint32_t)below, half);
    const uint32_t dmin_bits = half_reduce_min(__float_as_uint(dmin), half);
    const bool ok = !(__uint_as_float(dmin_bits) < MLB_WP_MARGIN * W);
    idx = idx > 127 ? 127 : idx;
    // p90 = np.percentile(values, 90) for n = 128: float32 'linear' rule of numpy >= 2 (same ops as features_ranked)
    const float vidx = 127.0f * (90.0f / 100.0f);
    const float fl = floorf(vidx);
    const int lo = (int)fl, hi = lo + 1;
    const float gamma = vidx - fl;
    const float a = vw[((lo & 7) << 4) | (lo >> 3)].x, b = vw[((hi & 7) << 4) | (hi >> 3)].x;
    const float p90_decay = vw[((idx & 7) << 4) | (idx >> 3)].x;
    const float diff = __fsub_rn(b, a);
    float p90 = __fadd_rn(a, __fmul_rn(diff, gamma));
    if (gamma >= 0.5f) p90 = __fsub_rn(b, __fmul_rn(diff, __fsub_rn(1.0f, gamma)));
    __syncwarp();  // scratch is reused by the next reservoir
    out[0] = mean;
    out[1] = p90;
    out[2] = sd;
    out[3] = mean_decay;
    out[4] = p90_decay;
    return ok;
}

// General incremental rank update on 8 slots per lane (packed ranks, SWAR): up to three written slots
// (7-bit ids in `list`), slots >= n_old are appends of the fill phase.  pm0 / pm1 carry one 0x01 per PRESENT
// slot; first every replaced slot's old rank is taken out, then the new values are inserted one at a time.
// The two halves of the warp may have different nchg: the loops run to the larger one with the shorter
// half predicated off, so that every collective is executed by the whole warp.
__device__ __forceinline__ void rank_update_h16(const float (&v)[8], uint32_t (&rkp)[2], uint32_t list, int nchg,
                                                int n_old, int hl, int half) {
    const int s0 = hl * 8;
    uint32_t pm0 = 0, pm1 = 0;
#pragma unroll
    for (int r = 0; r < 4; r++) {
        pm0 |= (s0 + r < n_old) ? (1u << (8 * r)) : 0u;
        pm1 |= (s0 + 4 + r < n_old) ? (1u << (8 * r)) : 0u;
    }
#pragma unroll 1
    for (int k = 0; k < 3; k++) {
        const int c = (list >> (7 * k)) & 127;
        const bool rem = k < nchg && c < n_old;
        if (!__any_sync(MLB_FULL, rem)) continue;
        const int sub = c & 7, lc = c >> 3;
        const uint32_t wsel = (sub & 4) ? rkp[1] : rkp[0];
        const uint32_t r_old = (__shfl_sync(MLB_FULL, wsel, lc, 16) >> (8 * (sub & 3))) & 255u;
        const uint32_t rep = ((r_old & 127u) + 1u) * 0x01010101u;
        const uint32_t g0 = ((((rkp[0] | 0x80808080u) - rep) >> 7) & pm0);
        const uint32_t g1 = ((((rkp[1] | 0x80808080u) - rep) >> 7) & pm1);
        if (rem) {
            rkp[0] -= g0;
            rkp[1] -= g1;
            if (hl == lc) {
                if (sub & 4) pm1 &= ~(1u << (8 * (sub & 3))); else pm0 &= ~(1u << (8 * (sub & 3)));
            }
        }
    }
#pragma unroll 1
    for (int k = 0; k < 3; k++) {
        const bool ins = k < nchg;
        if (!__any_sync(MLB_FULL, ins)) break;
        const int c = (list >> (7 * k)) & 127;
        const int sub = c & 7, lc = c >> 3;
        const float x = __shfl_sync(MLB_FULL, pick8(v, sub), lc, 16) + 0.0f;
        const uint32_t xb = __float_as_uint(x);
        const float xup = __uint_as_float((xb >> 31) ? xb - 1u : xb + 1u);
        uint32_t bef0 = 0, bef1 = 0;      // v_i <= x; slot c itself is not present yet (masked by pm below)
#pragma unroll
        for (int r = 0; r < 4; r++) {
            bef0 |= v[r] < xup ? (1u << (8 * r)) : 0u;
            bef1 |= v[r + 4] < xup ? (1u << (8 * r)) : 0u;
        }
        const uint32_t r_new = half_reduce_add_u16((uint32_t)(__popc(bef0 & pm0) + __popc(bef1 & pm1)), half);
        if (ins) {
            rkp[0] += ~bef0 & pm0;
            rkp[1] += ~bef1 & pm1;
            if (hl == lc) {
                const int sh = 8 * (sub & 3);
                if (sub & 4) { rkp[1] = (rkp[1] & ~(255u << sh)) | (r_new << sh); pm1 |= 1u << sh; }
                else { rkp[0] = (rkp[0] & ~(255u << sh)) | (r_new << sh); pm0 |= 1u << sh; }
            }
        }
    }
}

// features_ranked<4, false> on 8 slots per lane, returning false like features_full_h16: n valid slots (1..128),
// possibly different in the two halves
__device__ __forceinline__ bool features_any_h16(const float (&v)[8], const float (&t)[8], const uint32_t (&rkp)[2],
                                                 int n, float log2_decay, float2* vw, int hl, int half,
                                                 float (&out)[5]) {
    const int s0 = hl * 8;
    float s = 0.f, tm = -MLB_INF;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const bool valid = s0 + r < n;
        s += valid ? v[r] : 0.f;
        tm = valid ? fmaxf(tm, t[r]) : tm;
    }
    const float nf = (float)n;
    const float mean = half_sum(s) / nf;
    const float tmax = f32_from_orderable(half_reduce_max(f32_orderable(tm), half));
    float s2 = 0.f, svw = 0.f;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const bool valid = s0 + r < n;
        const float dv = v[r] - mean;
        s2 += valid ? dv * dv : 0.f;
        const float w = valid ? fast_exp2(log2_decay * (tmax - t[r])) : 0.f;
        svw += valid ? v[r] * w : 0.f;
        const uint32_t pos = valid ? ((rkp[r >> 2] >> (8 * (r & 3))) & 127u) : (uint32_t)(s0 + r);
        vw[((pos & 7u) << 4) | (pos >> 3)] = make_float2(v[r], w);
    }
    const float sd = fast_sqrt(half_sum(s2) / nf);
    svw = half_sum(svw);
    __syncwarp();
    float cum[8];
    float sw = 0.f;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        sw += vw[r * 16 + hl].y;
        cum[r] = sw;
    }
    float incl = sw;
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) {
        const float y = __shfl_up_sync(MLB_FULL, incl, o, 16);
        if (hl >= o) incl += y;
    }
    const float W = __shfl_sync(MLB_FULL, incl, 15, 16);
    const float mean_decay = svw * fast_rcp(W);
    const float rel = 0.9f * W - (incl - sw);
    int below = 0;
    float dmin = MLB_INF;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const bool valid = s0 + r < n;  // here s0 + r is a POSITION in rank order
        below += (valid && cum[r] < rel) ? 1 : 0;
        dmin = valid ? fminf(dmin, fabsf(cum[r] - rel)) : dmin;
    }
    int idx = (int)half_reduce_add_u16((uint32_t)below, half);
    const uint32_t dmin_bits = half_reduce_min(__float_as_uint(dmin), half);
    const bool ok = !(__uint_as_float(dmin_bits) < MLB_WP_MARGIN * W);
    idx = idx > n - 1 ? n - 1 : idx;
    const float vidx = (float)(n - 1) * (90.0f / 100.0f);
    const float fl = floorf(vidx);
    int lo = (int)fl, hi = lo + 1;
    if (vidx >= (float)(n - 1)) { lo = n - 1; hi = n - 1; }
    hi = hi > n - 1 ? n - 1 : hi;
    const float gamma = vidx - fl;
    const float a = vw[((lo & 7) << 4) | (lo >> 3)].x, b = vw[((hi & 7) << 4) | (hi >> 3)].x;
    const float p90_decay = vw[((idx & 7) << 4) | (idx >> 3)].x;
    const float diff = __fsub_rn(b, a);
    float p90 = __fadd_rn(a, __fmul_rn(diff, gamma));
    if (gamma >= 0.5f) p90 = __fsub_rn(b, __fmul_rn(diff, __fsub_rn(1.0f, gamma)));
    __syncwarp();
    out[0] = mean;
    out[1] = p90;
    out[2] = sd;
    out[3] = mean_decay;
    out[4] = p90_decay;
    return ok;
}

// lane q < 5 keeps feature q (the lane that stores it); lane 5 gets 1 when p90_decay sits on an exact tie
__device__ __forceinline__ float feature_of_lane(const float (&f)[5], bool tie, int lane) {
    float mine = f[0];
#pragma unroll
    for (int q = 1; q < 5; q++) mine = lane == q ? f[q] : mine;
    return lane == 5 ? (tie ? 1.f : 0.f) : mine;
}

// Returns feature `lane` in lanes 0..4, the exact-tie flag in lane 5.
static __device__ __noinline__ float warp_features_sorted(const float* __restrict__ vals, const float* __restrict__ tss,
                                                          uint8_t* __restrict__ ranks, int n, float now, double decay,
                                                          float log2_decay, float2* scratch) {
    const WarpScratch sc{scratch};
    float f[5];
    bool tie = false;
    if (n <= 0) {  // reservoir.py:127-134
#pragma unroll
        for (int q = 0; q < 5; q++) f[q] = 0.f;
    } else if (n <= 32) {
        features_sorted_epl<1>(vals, tss, ranks, n, now, decay, log2_decay, sc, f, tie);
    } else if (n <= 64) {
        features_sorted_epl<2>(vals, tss, ranks, n, now, decay, log2_decay, sc, f, tie);
    } else {
        features_sorted_epl<4>(vals, tss, ranks, n, now, decay, log2_decay, sc, f, tie);
    }
    return feature_of_lane(f, tie, lane_id());
}

// Ranks in global memory are valid (an incremental kernel updated and stored them) but its float32
// weighted-percentile decision was not trusted: evaluate from the stored ranks with the float64 tiers,
// no re-sort.  128-slot stride.  Returns feature `lane` in lanes 0..4, the exact-tie flag in lane 5.
static __device__ __noinline__ float warp_features_ranked_exact(const float* __restrict__ vals, const float* __restrict__ tss,
                                                                const uint8_t* __restrict__ ranks, int n, float now,
                                                                double decay, float log2_decay, float2* scratch) {
    const WarpScratch sc{scratch};
    const int lane = lane_id();
    float v[4], t[4], f[5];
    int rk[4];
    load_slots<4>(vals, lane, v);
    load_slots<4>(tss, lane, t);
    load_ranks<4>(ranks, lane, rk);
    bool tie;
    features_ranked<4, false>(v, t, rk, n, now, decay, log2_decay, sc, f, tie);
    return feature_of_lane(f, tie, lane);
}

}  // namespace mlb
