// The env step as two kernels, one warp per (env, LB agent) in both.
//
// Stands in for LoadBalanceEnv.step (reference:
// simulation-mode/problem-03-rl-environment/src/env.py:215-286) executed for
// E envs at once, with the flow-level dynamics of SURVEY.md App. B.
//
// event_kernel  (integer / pointer-chasing work, latency-bound)
//   phase 0  action -> weights (env.py:334-353); per-server scalars -> shared memory
//   phase A  per arrival (time order): retire finished flows (n_flow_on--, fct
//            sample -> Algorithm-R add, reservoir.py:50-85), choose a server
//            (SED / LSQ / power-of-two SED2, LSQ2 / alias, src/vpp/lb/node.c:393-460) with REDUX argmin,
//            push on that server's FIFO ring; the window end is one more
//            (pseudo-)event of the same loop
//   phase C  one flow_duration sample per still-active flow, state write-back,
//            one "changed slots" word per reservoir for the feature kernel
// feature_kernel  (float work, streams the touched reservoirs)
//   phase B  reservoir statistics of every reservoir touched this step
//            (reservoir.py:105-196) -> obs columns (features.py:256-286)
//   phase R  reward over the env's active servers (rewards.py:329-381), done flag
//
// Lane (server % 32) of the agent's warp owns every scalar of that server, so
// phases A/C need no intra-warp locking.  What is tested on every arrival (the
// finish time of the oldest flow, the assignment score) lives in registers,
// R = ceil(Sa/32) per lane; what changes only on events lives in shared memory.
// Phase B is warp-cooperative per reservoir with warp-uniform control flow.
// The split keeps each kernel's live state inside 64 registers (32 resident
// warps per SM) and each hot loop inside the instruction cache.
#pragma once
#include "mlb_common.cuh"
#include "mlb_env.cuh"
#include "mlb_features.cuh"
#include "../../include/marllb_b200.h"

namespace mlb {

// ---- event kernel: per-server shared-memory fields (4 bytes each), field f of server j at smem[f*SP + j]
enum : int {
    F_NON = 0,   // n_flow_on
    F_LASTFIN,   // finish time of the newest queued flow
    F_HEAD,      // ring position of the oldest in-system flow
    F_ACT,       // discrete action index (or float weight bits for continuous actions)
    F_CNT0, F_CNT1,  // reservoir counts   (fct, flow_duration)
    F_CUR0, F_CUR1,  // MT19937 replay cursors
    F_CHG0, F_CHG1,  // changed-slot word of each reservoir (see chg_* below)
    F_SPEED,     // processing speed
    NF
};

// "changed slots" word of one reservoir, event kernel -> feature kernel:
//   [0:7) [7:14) [14:21)  the first three distinct slots Algorithm R wrote this step
//   [21:24)               how many distinct slots were written (saturates at 7; > 3: re-sort)
//   [24:32)               n_old = valid slots at step start
__device__ __forceinline__ uint32_t chg_count(uint32_t w) { return (w >> 21) & 7u; }
__device__ __forceinline__ uint32_t chg_nold(uint32_t w) { return w >> 24; }

__host__ __device__ inline size_t event_warp_smem_bytes(int SP, bool alias) {
    return (size_t)NF * SP * 4 + (alias ? (size_t)SP * (8 + 4 + 8 + 4) : 0);
}

// ---- feature kernel: per-warp shared memory = dirty list | rank-order scratch
__host__ __device__ inline size_t feature_warp_smem_bytes(int SP) {
    return (size_t)2 * SP * 8 + MLB_SCRATCH_BYTES;
}

// Assignment score of one server as an order-preserving uint.
// node.c:395-404: f32 score = (n_flow_on + 1) / (1e-9 + weight), evaluated in double.
// For discrete actions the quotient comes from a table built on the host with exactly
// that arithmetic, stored in its order-preserving uint form: sed_table[a * (Q + 2) + n]; `act` is the row offset.
template <int POLICY>
__device__ __forceinline__ uint32_t server_score(const DevState& d, int n, uint32_t act) {
    if (POLICY == MLB_POLICY_SED || POLICY == MLB_POLICY_SED2) {
        if (d.action_kind == MLB_ACTION_CONTINUOUS_F32) {
            const double s = (double)(n + 1) / (1e-9 + (double)__uint_as_float(act));
            return f32_orderable((float)s);
        }
        return __ldg(d.sed_table + act + n);   // the table holds order-preserving uints; act = row offset a * (Q + 2)
    } else {
        return (uint32_t)n;  // node.c:419-431 (LSQ), :433-441 (LSQ2): f32(n) compares like n for 0 <= n <= Q
    }
}

// Index draw of ReservoirSampler.add (reservoir.py:65-85): returns the slot the
// sample goes to, or -1 when Algorithm R rejects it.  Replays
// RandomState(seed).randint(0, count+1): masked rejection over the raw MT19937
// words of that seed's row, `cur` = words consumed so far.
__device__ __forceinline__ int res_draw_slot(uint32_t cnt, uint32_t& cur, const uint32_t* __restrict__ row,
                                             int L, int K, int* status) {
    if (cnt < (uint32_t)K) return (int)cnt;  // fill phase, reservoir.py:65-73
    const uint32_t mask = 0xffffffffu >> __clz(cnt);
    uint32_t c = cur, v;
    do {
        if (c >= (uint32_t)L) {
            atomicOr(status, ST_ERR_RNG);
            v = 0xffffffffu;
            break;
        }
        v = __ldg(row + c) & mask;
        c++;
    } while (v > cnt);
    cur = c;
    return v < (uint32_t)K ? (int)v : -1;  // reservoir.py:78-85
}

// Philox4x32-10 (Salmon et al., SC'11), the counter-based generator of rng_mode = MLB_RNG_PHILOX.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint32_t (&out)[4]) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// Word `c` of the index stream of (global env g, server j): the stream every reservoir of that server draws from
// (both metrics: the reference hands the same seed to every metric's sampler, reservoir.py:261-265), each with its
// own cursor.  Twin: ora_philox_word in oracle/flow_oracle.c.  Out of line: the 10 rounds would otherwise be inlined
// at both add sites of the event kernel.
#define MLB_PHILOX_TAG 0x52535652u   /* "RSVR" */
#define MLB_PHILOX_KEY1 0x4d4c4232u  /* "MLB2" */
static __device__ __noinline__ uint32_t philox_stream_word(uint32_t c, uint32_t j, uint32_t g, uint32_t key0) {
    uint32_t r[4];
    philox4x32_10(c >> 2, j, g, MLB_PHILOX_TAG, key0, MLB_PHILOX_KEY1, r);
    const uint32_t lo = (c & 1u) ? r[1] : r[0], hi = (c & 1u) ? r[3] : r[2];
    return (c & 2u) ? hi : lo;
}

// res_draw_slot for rng_mode = MLB_RNG_PHILOX: the same masked-rejection rule (numpy's randint(0, count+1)) over the
// counter-based stream; no table, no length cap.
__device__ __forceinline__ int res_draw_slot_philox(uint32_t cnt, uint32_t& cur, uint32_t j, uint32_t g, uint32_t key0, int K) {
    if (cnt < (uint32_t)K) return (int)cnt;  // fill phase, reservoir.py:65-73
    const uint32_t mask = 0xffffffffu >> __clz(cnt);
    uint32_t c = cur, v;
    do {
        v = philox_stream_word(c, j, g, key0) & mask;
        c++;
    } while (v > cnt);
    cur = c;
    return v < (uint32_t)K ? (int)v : -1;  // reservoir.py:78-85
}

// per-warp view of the global arrays (32-bit offsets below these bases)
// 32-bit element offsets from the array bases in the kernel parameters (which live in the constant bank, not
// in registers): the event kernel is register-starved at 48 resident warps per SM
struct WarpGlobals {
    uint32_t res4;      // this agent's reservoirs [Sa][2][KP], in units of 4 floats (mlb_create checks the range)
    uint32_t ring;      // [Sa][Q] (arrival, finish) float2 index
    uint32_t mt;        // replay rows of this agent's servers [Sa][L]; philox mode: index of the agent's first server
    uint32_t genv;      // philox mode: global env id
};

// ReservoirSampler.add by the owning lane of server j, metric m.
template <int SP, int RNG>
__device__ __forceinline__ void res_add(const DevState& d, uint32_t* sm, const WarpGlobals& g, int m, int j,
                                        float value, float ts) {
    const uint32_t cnt = sm[(F_CNT0 + m) * SP + j];
    uint32_t c = sm[(F_CUR0 + m) * SP + j];
    const int slot = RNG == MLB_RNG_PHILOX
                         ? res_draw_slot_philox(cnt, c, g.mt + (uint32_t)j, g.genv, d.rng_key, d.K)
                         : res_draw_slot(cnt, c, d.mt_table + ((size_t)g.mt + (size_t)j * d.L), d.L, d.K, d.status);
    sm[(F_CUR0 + m) * SP + j] = c;
    sm[(F_CNT0 + m) * SP + j] = cnt + 1;
    if (slot >= 0) {
        const int at = (j * 2 + m) * d.KP + slot;
        const size_t ga = ((size_t)g.res4 << 2) + (size_t)at;
        d.res_val[ga] = value;
        d.res_ts[ga] = ts;
        // remember which slot changed (first three distinct ones; more -> ranks are re-sorted)
        uint32_t w = sm[(F_CHG0 + m) * SP + j];
        const uint32_t nc = chg_count(w);
        const bool dup = (nc >= 1 && (w & 127u) == (uint32_t)slot) || (nc >= 2 && ((w >> 7) & 127u) == (uint32_t)slot) ||
                         (nc >= 3 && ((w >> 14) & 127u) == (uint32_t)slot);
        if (!dup && nc < 7u) {
            if (nc < 3u) w |= (uint32_t)slot << (7 * nc);
            sm[(F_CHG0 + m) * SP + j] = w + (1u << 21);
        }
    }
}

// numpy pairwise block sum (n <= 128) and its two-block extension (n <= 256)
static __device__ inline double np_block_sum(const double* a, int n) {
    if (n < 8) {
        double r = -0.0;
        for (int i = 0; i < n; i++) r += a[i];
        return r;
    }
    double r[8];
    for (int k = 0; k < 8; k++) r[k] = a[k];
    int i;
    for (i = 8; i < n - (n % 8); i += 8)
        for (int k = 0; k < 8; k++) r[k] += a[i + k];
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; i++) res += a[i];
    return res;
}
static __device__ inline double np_sum_f64(const double* a, int n) {
    if (n <= 128) return np_block_sum(a, n);
    int n2 = n / 2;
    n2 -= n2 % 8;
    return np_block_sum(a, n2) + np_block_sum(a + n2, n - n2);
}

// rl_controller.py:359-405 _build_alias_table over p = w / sum(w); one lane.
static __device__ __noinline__ void alias_build(double* prob, int32_t* alias, int32_t* stack, const float* weight, int Sa) {
    for (int k = 0; k < Sa; k++) prob[k] = (double)weight[k];
    const double tot = np_sum_f64(prob, Sa);
    int* small = stack;
    int* large = stack + Sa;
    int ns = 0, nl = 0;
    for (int k = 0; k < Sa; k++) {
        const double p = (prob[k] / tot) * (double)Sa;
        prob[k] = p;
        alias[k] = k;
        if (p < 1.0) small[ns++] = k; else large[nl++] = k;
    }
    while (ns > 0 && nl > 0) {
        const int l = small[--ns];
        const int g = large[--nl];
        alias[l] = g;
        const double pg = prob[g] + prob[l] - 1.0;
        prob[g] = pg;
        if (pg < 1.0) small[ns++] = g; else large[nl++] = g;
    }
}

// Reward metric over staged reward-field values (one warp).
// rewards.py:21-287 and the original fair_fn table src/lb/env.py:73-156; float64 throughout like the reference.
template <typename T>
__device__ __noinline__ double reward_staged(int metric, const T* rv, const uint32_t* ra, int S) {
    const int lane = lane_id();
    const double eps = 1e-10;
    int na = 0;
    double sum = 0.0, sumsq = 0.0, mx = -1.0e308, mn = 1.0e308, slog = 0.0;
    for (int i = lane; i < S; i += 32) {
        if (!ra || ra[i]) {
            const double x = (double)rv[i];
            na++;
            sum += x;
            sumsq += x * x;
            mx = fmax(mx, x);
            mn = fmin(mn, x);
            if (metric == MLB_REWARD_PRODUCT) slog += log(x + eps);
        }
    }
    na = __reduce_add_sync(MLB_FULL, na);
    if (na == 0) return 0.0;  // rewards.py:364-365
    const double n = (double)na;
    sum = warp_sum(sum);
    switch (metric) {
    case MLB_REWARD_JAIN: {
        if (sum < eps) return 1.0;
        sumsq = warp_sum(sumsq);
        if (sumsq < eps) return 1.0;
        const double j = (sum * sum) / (n * sumsq);
        return fmin(fmax(j, 1.0 / n), 1.0);
    }
    case MLB_REWARD_FAIR_JAIN: {                        // src/lb/env.py:73-85: no clipping, guard is sum != 0
        if (sum == 0.0) return 1.0;
        return (sum * sum) / (n * warp_sum(sumsq));
    }
    case MLB_REWARD_FAIR_PRODUCT: {                     // src/lb/env.py:87-96
        const double den = warp_max(mx) + 1e-6;
        double p = 1.0;
        for (int i = lane; i < S; i += 32)
            if (!ra || ra[i]) p *= (double)rv[i] / den;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) p *= __shfl_xor_sync(MLB_FULL, p, o);
        return p;
    }
    case MLB_REWARD_MAX: return -warp_max(mx);
    case MLB_REWARD_MAX_EXP: return exp(-10000.0 * warp_max(mx));   // src/lb/env.py:142-149
    case MLB_REWARD_MAX_LOG: return -log(warp_max(mx));             // src/lb/env.py:135-139
    case MLB_REWARD_MIN: return warp_min(mn);
    case MLB_REWARD_RANGE: return -(warp_max(mx) - warp_min(mn));
    case MLB_REWARD_PRODUCT: return warp_sum(slog);
    default: break;
    }
    const double mean = sum / n;
    if (metric == MLB_REWARD_GINI) {
        if (mean == 0.0) return 0.0;
        double ds = 0.0;
        for (int i = lane; i < S; i += 32) {
            if (ra && !ra[i]) continue;
            const double xi = (double)rv[i];
            for (int k = 0; k < S; k++)
                if (!ra || ra[k]) ds += fabs(xi - (double)rv[k]);
        }
        ds = warp_sum(ds);
        return -(ds / (2.0 * n * n * mean));
    }
    double ss = 0.0;  // two-pass variance like np.var
    for (int i = lane; i < S; i += 32) {
        if (!ra || ra[i]) {
            const double dlt = (double)rv[i] - mean;
            ss += dlt * dlt;
        }
    }
    const double var = warp_sum(ss) / n;
    if (metric == MLB_REWARD_VARIANCE) return -var;
    if (metric == MLB_REWARD_STD) return -sqrt(var);
    if (metric == MLB_REWARD_VAR_EXP) return exp(-10000.0 * var);   // src/lb/env.py:108-115
    if (metric == MLB_REWARD_VAR_LOG) return -log(var);             // src/lb/env.py:118-125
    // MLB_REWARD_CV
    if (mean < eps) return 0.0;
    return -(sqrt(var) / (mean + eps));
}

// ---------------------------------------------------------------------------
// event_kernel: R = servers per lane (Sa <= 32*R), SP = 32*R.  Warps are independent.
constexpr int EV_MIN_BLOCKS = 10;   // resident blocks per SM the registers are budgeted for (40 warps)
template <int POLICY, int R, int RNG>
__global__ void __launch_bounds__(128, EV_MIN_BLOCKS)
event_kernel(const __grid_constant__ DevState d, const void* __restrict__ action) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int SP = 32 * R;
    constexpr bool kAlias = (POLICY == MLB_POLICY_ALIAS);
    // power of two choices (node.c:409-417, 433-441): two candidates from a pre-drawn bucket
    constexpr bool kPo2 = (POLICY == MLB_POLICY_SED2 || POLICY == MLB_POLICY_LSQ2);
    constexpr bool kArgmin = !kAlias && !kPo2;      // scan over all servers: scores live in registers
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int A = d.A, Sa = d.Sa, S = d.S;
    const int ea = d.e0 * A + blockIdx.x * (blockDim.x >> 5) + warp;
    if (ea >= d.e1 * A) return;
    const int e = ea / A;
    const int agent = ea - e * A;

    const size_t wbytes = event_warp_smem_bytes(SP, kAlias);
    unsigned char* wbase = smem_raw + (size_t)warp * wbytes;
    uint32_t* sm = reinterpret_cast<uint32_t*>(wbase);
    float* smf = reinterpret_cast<float*>(wbase);
    double* a_prob = reinterpret_cast<double*>(wbase + (size_t)NF * SP * 4);
    int32_t* a_alias = reinterpret_cast<int32_t*>(a_prob + SP);   // [SP] alias + [2*SP] builder stack
    float* a_w = reinterpret_cast<float*>(a_alias + 3 * SP);      // [SP] weights

    const int step = d.step[e] + 1;                       // env.py:230
    const float t1 = __fmul_rn((float)step, d.dt);        // window end
    const size_t sbase = (size_t)e * S + (size_t)agent * Sa;
    const int seed0 = agent * Sa;                         // replay row = server index in env
    WarpGlobals g;
    g.res4 = (uint32_t)(sbase * 2 * (d.KP >> 2));
    g.ring = (uint32_t)(sbase * d.Q);
    g.mt = RNG == MLB_RNG_PHILOX ? (uint32_t)seed0 : (uint32_t)((size_t)seed0 * d.L);
    g.genv = (uint32_t)(d.env_id_base + e);
    const int Q = d.Q;

    // ---------------- phase 0: load state, action -> weights -----------------
    float hf[R];       // finish time of the oldest in-system flow (INF: idle)
    float ha[R];       // its arrival time
    uint32_t sc[R];    // assignment score as an order-preserving uint
    static_for<R>([&](auto rc) {
        constexpr int r = decltype(rc)::value;
        const int j = lane + 32 * r;
        hf[r] = MLB_INF;
        ha[r] = 0.f;
        sc[r] = 0xffffffffu;
        if (j < Sa) {
            const size_t gi = sbase + j;
            const int n = d.n_on[gi];
            const uint32_t h = d.head[gi];
            sm[F_NON * SP + j] = (uint32_t)n;
            smf[F_LASTFIN * SP + j] = d.last_fin[gi];
            sm[F_HEAD * SP + j] = h;
            smf[F_SPEED * SP + j] = d.speed[gi];
            if (n > 0) {
                const float2 hd = d.ring[g.ring + j * Q + h];
                ha[r] = hd.x;
                hf[r] = hd.y;
                if (n > 1) prefetch_l2(d.ring + (g.ring + j * Q + (h + 1 == (uint32_t)Q ? 0u : h + 1)));
            }
            uint32_t act;
            if (d.action_kind == MLB_ACTION_CONTINUOUS_F32) {
                const float x = reinterpret_cast<const float*>(action)[gi];
                act = __float_as_uint(fminf(fmaxf(x, d.min_w), d.max_w));  // env.py:349-351
            } else {
                int a = d.action_kind == MLB_ACTION_DISCRETE_U8
                            ? (int)reinterpret_cast<const uint8_t*>(action)[gi]
                            : reinterpret_cast<const int32_t*>(action)[gi];
                if ((unsigned)a >= (unsigned)d.n_discrete) {
                    atomicOr(d.status, ST_ERR_ACTION);
                    a = 0;
                }
                // env.py:346; the SED policies keep the row offset into the score table instead of the index
                act = (POLICY == MLB_POLICY_SED || POLICY == MLB_POLICY_SED2) ? (uint32_t)(a * (Q + 2)) : (uint32_t)a;
            }
            sm[F_ACT * SP + j] = act;
            if (kArgmin) sc[r] = server_score<POLICY>(d, n, act);
#pragma unroll
            for (int m = 0; m < 2; m++) {
                const size_t c = ((size_t)e * 2 + m) * S + seed0 + j;
                const uint32_t cnt = d.res_count[c];
                sm[(F_CNT0 + m) * SP + j] = cnt;
                sm[(F_CUR0 + m) * SP + j] = d.res_cursor[c];
                sm[(F_CHG0 + m) * SP + j] = (cnt < (uint32_t)d.K ? cnt : (uint32_t)d.K) << 24;
            }
        }
    });
    __syncwarp();
    if (kAlias) {
        // weights as floats for the alias builder
        for (int j = lane; j < Sa; j += 32) {
            const uint32_t act = sm[F_ACT * SP + j];
            a_w[j] = d.action_kind == MLB_ACTION_CONTINUOUS_F32 ? __uint_as_float(act) : d.dw[act];
        }
        __syncwarp();
        if (lane == 0) alias_build(a_prob, a_alias, a_alias + SP, a_w, Sa);
        __syncwarp();
    }

    // ---------------- phase A: events of this window, in time order ----------
    const int64_t aoff = d.arr_off[ea];
    const int an = d.arr_n[ea];
    int cur = d.arr_cur[ea];
    for (;;) {
        const int idx = cur + lane;
        const float at = idx < an ? __ldcs(d.arr_time + aoff + idx) : MLB_INF;
        const unsigned bal = __ballot_sync(MLB_FULL, at < t1);
        const int nv = (bal == MLB_FULL) ? 32 : (__ffs(~bal) - 1);
        const bool last = nv < 32;
        const float awk = idx < an ? __ldcs(d.arr_work + aoff + idx) : 0.f;  // issued together with the times
        int abk = 0;
        float au = 0.f;
        if ((kAlias || kPo2) && lane < nv) {
            abk = __ldcs(d.arr_bucket + aoff + idx);
            if (kAlias) au = __ldcs(d.arr_u + aoff + idx);
        }
        const int iters = nv + (last ? 1 : 0);  // the window end is the final pseudo-event
        for (int i = 0; i < iters; i++) {
            const bool real = i < nv;
            const float ash = __shfl_sync(MLB_FULL, at, i & 31);
            const float wk = __shfl_sync(MLB_FULL, awk, i & 31);
            const float a = real ? ash : t1;
            // --- retire every flow that finished strictly before this event
            static_for<R>([&](auto rc) {
                constexpr int r = decltype(rc)::value;
                if (hf[r] < a) {
                    const int j = lane + 32 * r;
                    uint32_t h = sm[F_HEAD * SP + j];
                    int n = (int)sm[F_NON * SP + j];
                    float fin = hf[r], arr = ha[r];
                    do {
                        h = (h + 1 == (uint32_t)Q) ? 0u : h + 1;
                        n -= 1;                                             // src/vpp/lb/lbhash.h:120
                        float2 nx = make_float2(0.f, MLB_INF);
                        if (n > 0) nx = d.ring[g.ring + j * Q + h];          // in flight during the add
                        res_add<SP, RNG>(d, sm, g, 0, j, __fsub_rn(fin, arr), fin);  // lbhash.h:122-124
                        arr = nx.x;
                        fin = nx.y;
                    } while (fin < a);
                    hf[r] = fin;
                    ha[r] = arr;
                    sm[F_HEAD * SP + j] = h;
                    sm[F_NON * SP + j] = (uint32_t)n;
                    if (kArgmin) sc[r] = server_score<POLICY>(d, n, sm[F_ACT * SP + j]);
                }
            });
            __syncwarp();
            if (!real) break;
            // --- choose a server
            int kstar;
            if (kAlias) {
                const int b = __shfl_sync(MLB_FULL, abk, i);
                const float u = __shfl_sync(MLB_FULL, au, i);
                kstar = ((double)u < a_prob[b]) ? b : a_alias[b];           // test_integration.py:57-63
            } else if (kPo2) {
                // node.c:409-417 / 433-441: candidates = two consecutive flow-table entries; the second one
                // replaces the first only when its score is strictly lower.  Every lane evaluates both
                // (broadcast shared-memory reads), so no reduction is needed.
                const int c0 = __shfl_sync(MLB_FULL, abk, i);
                const int c1 = (c0 + 1 == Sa) ? 0 : c0 + 1;
                const uint32_t s0 = server_score<POLICY>(d, (int)sm[F_NON * SP + c0], sm[F_ACT * SP + c0]);
                const uint32_t s1 = server_score<POLICY>(d, (int)sm[F_NON * SP + c1], sm[F_ACT * SP + c1]);
                kstar = s1 < s0 ? c1 : c0;
            } else {
                uint32_t bkey = sc[0];
                int bj = lane;
                static_for<R>([&](auto rc) {
                    constexpr int r = decltype(rc)::value;
                    if (r > 0 && sc[r] < bkey) { bkey = sc[r]; bj = lane + 32 * r; }  // strict <: first minimum wins
                });
                const uint32_t mkey = __reduce_min_sync(MLB_FULL, bkey);
                kstar = (int)__reduce_min_sync(MLB_FULL, (uint32_t)(bkey == mkey ? bj : 0x7fffffff));
            }
            // --- push on that server's FIFO ring (owner lane)
            if (lane == (kstar & 31)) {
                const int k = kstar;
                const int n = (int)sm[F_NON * SP + k];
                if (n >= Q) {
                    atomicAdd(d.dropped + sbase + k, 1u);                   // [B] drop-and-count
                } else {
                    const float start = fmaxf(smf[F_LASTFIN * SP + k], a);
                    const float fin = __fadd_rn(start, __fdiv_rn(wk, smf[F_SPEED * SP + k]));
                    uint32_t pos = sm[F_HEAD * SP + k] + (uint32_t)n;
                    if (pos >= (uint32_t)Q) pos -= (uint32_t)Q;
                    d.ring[g.ring + k * Q + pos] = make_float2(a, fin);
                    smf[F_LASTFIN * SP + k] = fin;
                    sm[F_NON * SP + k] = (uint32_t)(n + 1);                 // lbhash.h:142,167
                    uint32_t nsc = 0;
                    if (kArgmin) nsc = server_score<POLICY>(d, n + 1, sm[F_ACT * SP + k]);
                    static_for<R>([&](auto rc) {
                        constexpr int r = decltype(rc)::value;
                        if ((k >> 5) == r) {
                            if (n == 0) { hf[r] = fin; ha[r] = a; }
                            sc[r] = nsc;
                        }
                    });
                }
                if (d.record_assign) d.assign[aoff + cur + i] = seed0 + k;
            }
            __syncwarp();
        }
        cur += nv;
        if (last) break;
    }
    if (lane == 0) d.arr_cur[ea] = cur;

    // ---------------- phase C: flow_duration samples, state write-back -------
    float* obs = d.obs + sbase * MLB_OBS_COLS;
    static_for<R>([&](auto rc) {
        constexpr int r = decltype(rc)::value;
        const int j = lane + 32 * r;
        if (j < Sa) {
            const size_t gi = sbase + j;
            const int n = (int)sm[F_NON * SP + j];
            uint32_t pos = sm[F_HEAD * SP + j];
            d.n_on[gi] = n;
            d.last_fin[gi] = smf[F_LASTFIN * SP + j];
            d.head[gi] = pos;
            obs[j * MLB_OBS_COLS] = (float)n;                               // features.py:274
            float arr = ha[r];  // the oldest flow is in registers
            for (int q = 0; q < n; q++) {  // lbhash.h:131-135, one sample per active flow per step
                pos = (pos + 1 == (uint32_t)Q) ? 0u : pos + 1;
                float nx = 0.f;
                if (q + 1 < n) nx = d.ring[g.ring + j * Q + pos].x;          // in flight during the add
                res_add<SP, RNG>(d, sm, g, 1, j, __fsub_rn(t1, arr), t1);
                arr = nx;
            }
#pragma unroll
            for (int m = 0; m < 2; m++) {
                const size_t c = ((size_t)e * 2 + m) * S + seed0 + j;
                d.res_count[c] = sm[(F_CNT0 + m) * SP + j];
                d.res_cursor[c] = sm[(F_CUR0 + m) * SP + j];
                d.res_chg[c] = sm[(F_CHG0 + m) * SP + j];
            }
        }
    });
}

// ---------------------------------------------------------------------------
// pair_kernel: the incremental statistics of every cached reservoir with a 128-slot stride (K = 97..128) whose
// stored ranks are valid and in which Algorithm R wrote 1..3 slots -- two reservoirs per warp instruction (one per
// half-warp, 8 slots per lane; see mlb_features.cuh).  One warp per (env, agent), warps independent.  A separate
// kernel so that its loop (~420 instructions per pair) has the instruction cache to itself: inside feature_kernel
// the two hot paths evicted each other (ncu: 29 % of the stalls were instruction fetches).
//
// Shared memory per warp: dirty list | two rank-order scratches | two staging buffers.  A staging buffer holds
// values[128] | timestamps[128] | ranks[128 bytes] of one reservoir of the NEXT pair, filled by cp.async while the
// current pair is being evaluated.
#define MLB_STAGE_BYTES 1152
__host__ __device__ inline size_t pair_warp_smem_bytes(int SP) {
    return (size_t)2 * SP * 8 + 2 * MLB_SCRATCH_BYTES + 2 * MLB_STAGE_BYTES;
}

// CLS 0: full reservoirs with ONE replaced slot (constants folded, one-slot SWAR update);
// CLS 1: every other incrementally updatable reservoir (2-3 written slots, fill-phase appends, K < 128).
template <int R, int CLS>
__global__ void __launch_bounds__(128, 8)
pair_kernel(const __grid_constant__ DevState d) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int SP = 32 * R;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int A = d.A, Sa = d.Sa, S = d.S;
    // Large launches: one warp per (env, agent).  Small ones (a few thousand envs: a fraction of a wave, where the time
    // is one warp's walk through its list) deal the list of one (env, agent) out to the four warps of a block.
    const int wpe = d.pair_wpe;
    const int ea = d.e0 * A + (wpe == 1 ? blockIdx.x * (blockDim.x >> 5) + warp : (int)blockIdx.x);
    const int sub = wpe == 1 ? 0 : warp;
    if (ea >= d.e1 * A) return;
    const int e = ea / A;
    const int agent = ea - e * A;
    unsigned char* wbase = smem_raw + (size_t)warp * pair_warp_smem_bytes(SP);
    uint2* dlist = reinterpret_cast<uint2*>(wbase);
    float2* const vw = reinterpret_cast<float2*>(wbase + (size_t)2 * SP * 8);
    unsigned char* stage = wbase + (size_t)2 * SP * 8 + 2 * MLB_SCRATCH_BYTES;
    const size_t sbase = (size_t)e * S + (size_t)agent * Sa;
    const int seed0 = agent * Sa;

    int nfast = 0;
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int j = lane + 32 * r;
#pragma unroll
        for (int m = 0; m < 2; m++) {
            uint32_t chg = 0, cnt = 0;
            if (j < Sa) {
                const size_t c = ((size_t)e * 2 + m) * S + seed0 + j;
                chg = __ldg(d.res_chg + c);
                cnt = __ldg(d.res_count + c);
            }
            const uint32_t nchg = chg_count(chg);
            const uint32_t n = cnt < (uint32_t)d.K ? cnt : (uint32_t)d.K;
            const bool one = nchg == 1 && chg_nold(chg) == 128 && n == 128;
            // n_old == 255: pair_kernel<.,0> could not settle this one and handed it to feature_kernel.  On small launches
            // the two pair kernels run side by side, so <.,1> may or may not see that mark yet -- either way the entry is
            // not its own ("one" before the mark, "redo" after it).
            const bool redo = chg_nold(chg) == 255u;
            const bool inc = !redo && chg_nold(chg) > 0 && nchg >= 1 && nchg <= 3;
            const bool fast = j < Sa && (CLS == 0 ? one : (inc && !one));
            const unsigned bal = __ballot_sync(MLB_FULL, fast);
            if (fast) dlist[nfast + __popc(bal & ((1u << lane) - 1u))] = make_uint2(chg, (uint32_t)(j * 2 + m) | (n << 9));
            nfast += __popc(bal);
        }
    }
    __syncwarp();
    if (nfast == 0) return;
    const float4* const val4 = reinterpret_cast<const float4*>(d.res_val);
    const float4* const ts4 = reinterpret_cast<const float4*>(d.res_ts);
    uint32_t* const rank4 = reinterpret_cast<uint32_t*>(d.res_rank);
    uint32_t off0 = (uint32_t)(sbase * 2 * 32) + (uint32_t)lane;
    uint32_t obs0 = (uint32_t)(sbase * MLB_OBS_COLS) + 1u;
    uint32_t chg0 = (uint32_t)((size_t)e * 2 * S + seed0);
    // opaque to the optimiser: otherwise they are re-derived from (env, agent) with 64-bit multiplies inside the loop
    // instead of living in three registers
    asm volatile("" : "+r"(off0), "+r"(obs0), "+r"(chg0));
    const uint32_t stage_s = (uint32_t)__cvta_generic_to_shared(stage) + lane * 16;
    const int half = lane >> 4, hl = lane & 15;
    float2* const vw_half = vw + half * 128;
    auto stage_in = [&](uint32_t id, int slot) {
        const uint32_t off = off0 + id * 32u;
        const uint32_t dst = stage_s + (uint32_t)slot * MLB_STAGE_BYTES;
        cp_async16(dst, val4 + off);
        cp_async16(dst + 512, ts4 + off);
        cp_async4(dst + 1024 - lane * 12, rank4 + off);
    };
    const int i0 = 2 * sub, di = 2 * wpe;     // this warp takes the pairs i0, i0 + di, ...
    if (i0 >= nfast) return;
    stage_in(dlist[i0].y & 511u, 0);
    if (i0 + 1 < nfast) stage_in(dlist[i0 + 1].y & 511u, 1);
    cp_async_commit();
#pragma unroll 1
    for (int i = i0; i < nfast; i += di) {
        const bool valid = i + half < nfast;              // an odd list ends with half 1 idle
        const uint2 ent = dlist[valid ? i + half : i];
        const uint32_t id = ent.y & 511u;
        cp_async_wait_all();
        __syncwarp();
        const unsigned char* rec = stage + half * MLB_STAGE_BYTES;
        const float4 v0 = reinterpret_cast<const float4*>(rec)[hl * 2], v1 = reinterpret_cast<const float4*>(rec)[hl * 2 + 1];
        const float4 t0 = reinterpret_cast<const float4*>(rec + 512)[hl * 2], t1q = reinterpret_cast<const float4*>(rec + 512)[hl * 2 + 1];
        const uint2 rq = reinterpret_cast<const uint2*>(rec + 1024)[hl];
        __syncwarp();
        if (i + di < nfast) {
            stage_in(dlist[i + di].y & 511u, 0);
            if (i + di + 1 < nfast) stage_in(dlist[i + di + 1].y & 511u, 1);
            cp_async_commit();
        }
        const float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
        const float t[8] = {t0.x, t0.y, t0.z, t0.w, t1q.x, t1q.y, t1q.z, t1q.w};
        uint32_t rkp[2] = {valid ? rq.x : 0u, valid ? rq.y : 0u};   // idle half: every scatter position 0
        float f[5];
        bool ok;
        if (CLS == 0) {
            rank_replace_one_h16(v, rkp, (int)(ent.x & 127u), hl, half);
            if (valid) reinterpret_cast<uint2*>(rank4 + (off0 - lane + id * 32u))[hl] = make_uint2(rkp[0], rkp[1]);
            if (!valid) { rkp[0] = 0u; rkp[1] = 0u; }
            ok = features_full_h16(v, t, rkp, d.log2_decay, vw_half, hl, half, f);
        } else {
            const int n = valid ? (int)((ent.y >> 9) & 255u) : 1;
            rank_update_h16(v, rkp, ent.x, valid ? (int)chg_count(ent.x) : 0, valid ? (int)chg_nold(ent.x) : 1, hl, half);
            if (valid) reinterpret_cast<uint2*>(rank4 + (off0 - lane + id * 32u))[hl] = make_uint2(rkp[0], rkp[1]);
            if (!valid) { rkp[0] = 0u; rkp[1] = 0u; }
            ok = features_any_h16(v, t, rkp, n, d.log2_decay, vw_half, hl, half, f);
        }
        if (valid && hl == 0) {
            if (ok) {
                float* o = d.obs + (obs0 + (id >> 1) * MLB_OBS_COLS + (id & 1u) * 5u);
#pragma unroll
                for (int q = 0; q < 5; q++) o[q] = f[q];
            } else {
                // float32 decision not trusted: hand the reservoir to feature_kernel (n_old = 255 marks "ranks are
                // valid, decide in float64"; [E][2][S] layout: metric-major)
                d.res_chg[chg0 + (id & 1u) * (uint32_t)S + (id >> 1)] = (ent.x & 0x00ffffffu) | (255u << 24);
            }
        }
    }
}

// ---------------------------------------------------------------------------
// feature_kernel: block = epb envs x A agent warps (the reward needs all agents of an env).
// SMALL: blocks of at most 128 threads (A * epb <= 4 warps), compiled for 48 resident warps per SM: what is left
// for this kernel once pair_kernel took the incremental entries is a latency chain per warp (list loads, the
// occasional re-sort, obs reads for the reward), hidden by residency rather than by instruction-level parallelism.
template <int R, bool SMALL>
__global__ void __launch_bounds__(SMALL ? 128 : 1024, SMALL ? 12 : 1)
feature_kernel(const __grid_constant__ DevState d) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int SP = 32 * R;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int A = d.A, Sa = d.Sa, S = d.S;
    const int nwarps = blockDim.x >> 5;
    const int epb = nwarps / A;
    const int env_in_blk = warp / A;
    const int agent = warp - env_in_blk * A;
    const int e = d.e0 + blockIdx.x * epb + env_in_blk;
    if (e >= d.e1) return;  // whole env (all its warps) leaves together

    // ---- shared memory: [per warp: dirty list | scratch] ... [per env: reward staging]
    const size_t wbytes = feature_warp_smem_bytes(SP);
    unsigned char* wbase = smem_raw + (size_t)warp * wbytes;
    uint2* dlist = reinterpret_cast<uint2*>(wbase);
    const WarpScratch scratch{reinterpret_cast<float2*>(wbase + (size_t)2 * SP * 8)};
    float* rv = reinterpret_cast<float*>(smem_raw + (size_t)nwarps * wbytes) + (size_t)env_in_blk * 2 * S;
    uint32_t* ra = reinterpret_cast<uint32_t*>(rv + S);

    const int step = d.step[e] + 1;                       // env.py:230
    const float t1 = __fmul_rn((float)step, d.dt);        // window end
    const size_t sbase = (size_t)e * S + (size_t)agent * Sa;
    const int seed0 = agent * Sa;
    float* const res_val = d.res_val + sbase * 2 * d.KP;
    float* const res_ts = d.res_ts + sbase * 2 * d.KP;
    uint8_t* const res_rank = d.res_rank + sbase * 2 * d.KP;
    float* const obs = d.obs + sbase * MLB_OBS_COLS;

    // ---------------- phase B: statistics of touched reservoirs --------------
    // The dirty (server, metric) pairs are first compacted into a list, every lane describing
    // its own servers: entry = { changed-slot word, id | n << 9 | redo << 18 }.
    const bool all = d.feature_cache == 0;  // mode 0: recompute every reservoir
    const int KP = d.KP;
    // Entries with valid stored ranks and 1..3 written slots were already evaluated by pair_kernel; an entry it
    // could not settle comes back with n_old = 255 ("redo": ranks valid, float64 decision needed).  This kernel
    // takes everything else.
    int nd = 0;
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int j = lane + 32 * r;
#pragma unroll
        for (int m = 0; m < 2; m++) {
            uint32_t chg = 0, cnt = 0;
            if (j < Sa) {
                const size_t c = ((size_t)e * 2 + m) * S + seed0 + j;
                chg = __ldg(d.res_chg + c);
                cnt = __ldg(d.res_count + c);
            }
            const uint32_t nchg = chg_count(chg);
            const uint32_t n = cnt < (uint32_t)d.K ? cnt : (uint32_t)d.K;
            const bool redo = chg_nold(chg) == 255u;
            const bool fast = d.use_pair && !redo && chg_nold(chg) > 0 && nchg >= 1 && nchg <= 3;
            const bool take = j < Sa && (all || nchg > 0) && !fast;
            const unsigned bal = __ballot_sync(MLB_FULL, take);
            if (take)
                dlist[nd + __popc(bal & ((1u << lane) - 1u))] =
                    make_uint2(chg, (uint32_t)(j * 2 + m) | (n << 9) | ((redo ? 1u : 0u) << 18));
            nd += __popc(bal);
        }
    }
    __syncwarp();
    float* const warp_obs = obs + 1;
#pragma unroll 1
    for (int i = 0; i < nd; i++) {
        const uint2 ent = dlist[i];
        const uint32_t id = ent.y & 511u;
        const int n = (int)((ent.y >> 9) & 255u);
        const int rid = (int)id * KP;
        float mine;
        if ((ent.y >> 18) & 1u)
            mine = warp_features_ranked_exact(res_val + rid, res_ts + rid, res_rank + rid, n, t1, d.decay,
                                              d.log2_decay, scratch.vw);
        else
            mine = warp_features_sorted(res_val + rid, res_ts + rid, res_rank + rid, n, t1, d.decay,
                                        d.log2_decay, scratch.vw);
        if (lane < 5) warp_obs[(id >> 1) * MLB_OBS_COLS + (id & 1u) * 5u + lane] = mine;
    }
    __syncwarp();

    // ---------------- phase R: reward over the env's active servers ----------
#pragma unroll 1
    for (int j = lane; j < Sa; j += 32) {
        const float* row = obs + j * MLB_OBS_COLS;
        bool active = false;  // env.py:410-413
        float x = 0.f;
#pragma unroll
        for (int c = 0; c < MLB_OBS_COLS; c++) {
            const float o = row[c];
            active |= o > 0.f;
            x = c == d.reward_field ? o : x;
        }
        rv[seed0 + j] = x;
        ra[seed0 + j] = active ? 1u : 0u;
    }
    if (A == 1) {
        __syncwarp();
    } else if (env_in_blk == 0) {  // at most 2 envs per block when A > 1: static barrier ids
        asm volatile("bar.sync 1, %0;" ::"r"(A * 32) : "memory");
    } else {
        asm volatile("bar.sync 2, %0;" ::"r"(A * 32) : "memory");
    }
    if (agent == 0) {
        const double rw = reward_staged<float>(d.reward_metric, rv, ra, S);
        if (lane == 0) {
            d.reward[e] = rw;                              // multi_agent_env.py:143-145: same scalar for all agents
            d.done[e] = step >= d.max_steps ? 1 : 0;       // env.py:267
            d.step[e] = step;
        }
    }
}

}  // namespace mlb
