// C ABI of the env path (include/marllb_b200.h): handle, device state, launches.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <new>
#include <string>
#include <vector>

#include "mlb_mt19937.h"
#include "mlb_step_kernel.cuh"

using namespace mlb;

struct mlb_env {
    mlb_config cfg;
    DevState d;
    int device = 0;
    std::string err;
    int64_t launches = 0;
    std::vector<void*> allocs;
    // arrival storage (owned)
    float *arr_time = nullptr, *arr_work = nullptr, *arr_u = nullptr;
    int32_t* arr_bucket = nullptr;
    int64_t* arr_off = nullptr;
    int32_t* arr_n = nullptr;
    int64_t arr_total = 0;
    std::vector<int64_t> h_off;
    std::vector<int32_t> h_n;
    bool have_arrivals = false;
    // staged (next) chunk of a streamed trace: filled asynchronously, swapped in by mlb_commit_arrivals
    float *stg_time = nullptr, *stg_work = nullptr, *stg_u = nullptr;
    int32_t* stg_bucket = nullptr;
    int64_t* stg_off = nullptr;
    int32_t* stg_n = nullptr;
    int64_t stg_total = 0;
    std::vector<int64_t> stg_h_off;
    std::vector<int32_t> stg_h_n;
    cudaEvent_t stg_ready = nullptr;   // staged copies done
    cudaEvent_t stg_free = nullptr;    // last kernel that read the buffers now used for staging has finished
    bool stg_pending = false, stg_valid = false;
    void* d_action = nullptr;
    size_t action_bytes = 0;
    uint8_t* d_mask = nullptr;
    size_t ev_smem = 0, ft_smem = 0, pr_smem = 0;   // dynamic shared memory of the event / feature / pair kernel
    // kernel instantiations of this config; pr_fn[c] = pair_kernel<R, c>
    const void *ev_fn = nullptr, *ft_fn = nullptr, *pr_fn[3] = {nullptr, nullptr, nullptr};
    bool use_pair = false;             // pair_kernel applies (128-slot reservoir stride, feature cache on)
    // large launches (> 8192 (env, agent) pairs) run both classes in one pair_kernel<.,2>; small ones run
    // pair_kernel<.,1> BESIDE pair_kernel<.,0> (disjoint reservoirs) on this stream -- under a stream capture a
    // parallel branch of the graph; at those sizes each launch is one warp's latency chain
    cudaStream_t pair_stream = nullptr;
    cudaEvent_t pair_fork = nullptr, pair_join = nullptr;
    int ev_threads = 128;              // event kernel: independent warps
    int epb = 1, ft_threads = 32;      // feature kernel: epb envs x A agent warps per block
    cudaStream_t copy_stream = nullptr;   // device->host copies of the chunked host-buffer step
    cudaEvent_t copy_done = nullptr;
    std::vector<cudaEvent_t> chunk_ev;
    int host_chunks = 8;
    std::vector<cudaEvent_t> prof_ev;  // 4 events per profiled step: | event | pair | feature |
    double prof_pair_ms = 0.0;         // pair_kernel share of the last mlb_profile_end
    int prof_cap = 0, prof_n = 0;
    size_t state_bytes[MLB_F_COUNT_] = {0};
    void* state_ptr[MLB_F_COUNT_] = {nullptr};
    // changed-rows host step (mlb_step_changed): device compaction buffers, pinned staging, host apply threads
    uint32_t* cr_rec = nullptr;        // device [E*S][12] records: row index | 11 floats
    uint16_t* cr_col = nullptr;        // device [E*S] n_flow_on column (dense, 2 bytes per row)
    uint32_t* cr_cnt = nullptr;        // device [chunks] records written per chunk
    uint32_t* cr_h_rec = nullptr;      // pinned mirrors
    uint16_t* cr_h_col = nullptr;
    uint32_t* cr_h_cnt = nullptr;
    std::vector<cudaEvent_t> cr_ev_cnt, cr_ev_copy;
    struct HostPool* pool = nullptr;
    // mlb_stage_arrivals may run on a second host thread next to mlb_step (see the header): the allocation list
    // and the error text are the two things both threads write
    std::mutex mu;
};

static std::string g_create_err;

static int fail(mlb_env* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) {
        std::lock_guard<std::mutex> lk(h->mu);
        h->err = buf;
    } else {
        g_create_err = buf;
    }
    return code;
}

#define CK(h, call)                                                                            \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return fail(h, MLB_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                        __FILE__, __LINE__);                                                   \
    } while (0)

template <typename T>
static cudaError_t dalloc(mlb_env* h, T** p, size_t n) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, n * sizeof(T) > 0 ? n * sizeof(T) : 16);
    if (e == cudaSuccess) {
        // debug aid (tools/determinism_probe.py): MLB_POISON=<byte> fills every fresh allocation, so that a read of
        // memory nothing wrote shows up as a difference between two runs with different fill bytes
        if (const char* pz = getenv("MLB_POISON")) e = cudaMemset(q, (int)strtol(pz, nullptr, 0) & 255, n * sizeof(T) > 0 ? n * sizeof(T) : 16);
    }
    if (e == cudaSuccess) {
        std::lock_guard<std::mutex> lk(h->mu);
        h->allocs.push_back(q);
        *p = reinterpret_cast<T*>(q);
    }
    return e;
}

// ------------------------------------------------------------------ kernels
__global__ void fill_f32_kernel(float* p, size_t n, float v) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        p[i] = v;
}

// speeds[S] (device) broadcast to every env's row of d.speed [E][S]
__global__ void bcast_rows_kernel(float* __restrict__ dst, const float* __restrict__ row, int S, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = __ldg(row + (int)(i % (size_t)S));
}

// reset(): zero every per-env slice of the selected envs (env.py:186-213;
// reservoir.py:220-225 zero-fills the sample arrays).  One block per env.
__global__ void reset_kernel(const DevState d, const uint8_t* __restrict__ mask) {
    const int e = blockIdx.x;
    if (mask && !mask[e]) return;
    const int S = d.S, tid = threadIdx.x, nt = blockDim.x;
    const size_t sb = (size_t)e * S;
    for (int i = tid; i < S; i += nt) {
        d.n_on[sb + i] = 0;
        d.last_fin[sb + i] = 0.f;
        d.head[sb + i] = 0;
        d.dropped[sb + i] = 0;
    }
    for (int i = tid; i < 2 * S; i += nt) {
        d.res_count[(size_t)e * 2 * S + i] = 0;
        d.res_cursor[(size_t)e * 2 * S + i] = 0;
        d.res_tie[(size_t)e * 2 * S + i] = 0;
    }
    const size_t rn = (size_t)S * 2 * d.KP;
    float4* v4 = reinterpret_cast<float4*>(d.res_val + sb * 2 * d.KP);
    float4* t4 = reinterpret_cast<float4*>(d.res_ts + sb * 2 * d.KP);
    uint32_t* r4 = reinterpret_cast<uint32_t*>(d.res_rank + sb * 2 * d.KP);
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    for (size_t i = tid; i < rn / 4; i += nt) {
        v4[i] = z;
        t4[i] = z;
        r4[i] = 0u;
    }
    for (int i = tid; i < S * MLB_OBS_COLS; i += nt) d.obs[sb * MLB_OBS_COLS + i] = 0.f;
    for (int i = tid; i < d.A; i += nt) d.arr_cur[(size_t)e * d.A + i] = 0;
    if (tid == 0) {
        d.reward[e] = 0.0;
        d.done[e] = 0;
        d.step[e] = 0;
    }
}

// One warp per (env, agent) stream: exponential inter-arrivals (rate/s) kept
// while < horizon, exponential work (training_pipeline.py:141-155 semantics).
__global__ void gen_poisson_kernel(float* __restrict__ time, float* __restrict__ work,
                                   int32_t* __restrict__ bucket, float* __restrict__ uu,
                                   int32_t* __restrict__ count, int n_streams, int cap, int Sa,
                                   uint32_t stream_base, double rate, double mean_work,
                                   double t_start, double horizon, uint64_t seed, uint32_t window) {
    const int lane = threadIdx.x & 31;
    const int sidx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (sidx >= n_streams) return;
    const size_t base = (size_t)sidx * cap;
    double t0 = t_start;
    int n = 0;
    for (int chunk = 0; n < cap && t0 < horizon; chunk++) {
        uint32_t r[4];
        philox4x32_10((uint32_t)(chunk * 32 + lane), stream_base + (uint32_t)sidx, 0x4d4c4221u, window,
                      (uint32_t)seed, (uint32_t)(seed >> 32), r);
        const double u1 = ((double)r[0] + 0.5) * (1.0 / 4294967296.0);
        const double u2 = ((double)r[1] + 0.5) * (1.0 / 4294967296.0);
        double dtv = -log(u1) / rate;
        // inclusive warp scan of inter-arrival gaps
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double y = __shfl_up_sync(MLB_FULL, dtv, o);
            if (lane >= o) dtv += y;
        }
        const double t = t0 + dtv;
        const bool keep = (t < horizon) && (n + lane < cap);
        if (keep) {
            time[base + n + lane] = (float)t;
            work[base + n + lane] = (float)(-log(u2) * mean_work);
            if (bucket) {
                bucket[base + n + lane] = (int32_t)(r[2] % (uint32_t)Sa);
                uu[base + n + lane] = (float)(r[3] >> 8) * (1.0f / 16777216.0f);
            }
        }
        n += __popc(__ballot_sync(MLB_FULL, keep));
        t0 = __shfl_sync(MLB_FULL, t, 31);
    }
    if (lane == 0) count[sidx] = n;
}

// ------------------------------------------------------------------ changed-rows compaction
// One thread per (env, server) row of envs [e0, e1): writes the row's n_flow_on into the dense 16-bit column and,
// when Algorithm R wrote a slot of either reservoir of the row this step (res_chg, written by event_kernel for
// every reservoir) or feature_kernel re-evaluated one of them as an exact tie (res_tie), appends {row index, the 11
// observation floats} to this chunk's record list.
__global__ void compact_rows_kernel(const DevState d, uint32_t* __restrict__ rec, uint16_t* __restrict__ col,
                                    uint32_t* __restrict__ cnt) {
    const int S = d.S;
    const size_t row0 = (size_t)d.e0 * S, rows = (size_t)(d.e1 - d.e0) * S;
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    const bool in = i < rows;
    const size_t row = row0 + (in ? i : 0);
    const int e = (int)(row / S), sv = (int)(row - (size_t)e * S);
    bool changed = false;
    if (in) {
        const uint32_t c0 = d.res_chg[((size_t)e * 2 + 0) * S + sv], c1 = d.res_chg[((size_t)e * 2 + 1) * S + sv];
        changed = d.feature_cache != 1 || ((c0 >> 21) & 7u) != 0u || ((c1 >> 21) & 7u) != 0u ||
                  d.res_tie[((size_t)e * 2 + 0) * S + sv] != 0 || d.res_tie[((size_t)e * 2 + 1) * S + sv] != 0;
        col[row] = (uint16_t)d.n_on[row];
    }
    const unsigned bal = __ballot_sync(MLB_FULL, changed);
    if (bal == 0u) return;
    const int lane = threadIdx.x & 31;
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(cnt, (uint32_t)__popc(bal));
    base = __shfl_sync(MLB_FULL, base, 0);
    if (changed) {
        const size_t k = row0 + base + __popc(bal & ((1u << lane) - 1u));   // chunk's region starts at its first row
        const float* o = d.obs + row * MLB_OBS_COLS;
        uint4* r = reinterpret_cast<uint4*>(rec + k * 12);
        r[0] = make_uint4((uint32_t)row, __float_as_uint(o[0]), __float_as_uint(o[1]), __float_as_uint(o[2]));
        r[1] = make_uint4(__float_as_uint(o[3]), __float_as_uint(o[4]), __float_as_uint(o[5]), __float_as_uint(o[6]));
        r[2] = make_uint4(__float_as_uint(o[7]), __float_as_uint(o[8]), __float_as_uint(o[9]), __float_as_uint(o[10]));
    }
}

// Host threads that apply the compact records to the caller's observation array (persistent across calls).
struct HostPool {
    std::vector<std::thread> th;
    std::mutex mu;
    std::condition_variable cv, cv_done;
    std::function<void(int, int)> job;
    uint64_t gen = 0;
    int pending = 0;
    bool stop = false;
    explicit HostPool(int n) {
        for (int t = 0; t < n; t++)
            th.emplace_back([this, t, n] {
                uint64_t seen = 0;
                for (;;) {
                    std::function<void(int, int)> f;
                    {
                        std::unique_lock<std::mutex> lk(mu);
                        cv.wait(lk, [&] { return stop || gen != seen; });
                        if (stop) return;
                        seen = gen;
                        f = job;
                    }
                    f(t, n);
                    std::lock_guard<std::mutex> lk(mu);
                    if (--pending == 0) cv_done.notify_all();
                }
            });
    }
    void run(std::function<void(int, int)> f) {      // f(thread index, thread count) on every thread; returns when all are done
        std::unique_lock<std::mutex> lk(mu);
        job = std::move(f);
        pending = (int)th.size();
        gen++;
        cv.notify_all();
        cv_done.wait(lk, [&] { return pending == 0; });
    }
    ~HostPool() {
        {
            std::lock_guard<std::mutex> lk(mu);
            stop = true;
        }
        cv.notify_all();
        for (auto& t : th) t.join();
    }
};

// ------------------------------------------------------------------ helpers
template <int POLICY, int RNG>
static const void* event_fn_r(int R) {
    switch (R) {
    case 1: return (const void*)event_kernel<POLICY, 1, RNG>;
    case 2: return (const void*)event_kernel<POLICY, 2, RNG>;
    case 4: return (const void*)event_kernel<POLICY, 4, RNG>;
    default: return (const void*)event_kernel<POLICY, 8, RNG>;
    }
}
static int lanes_r(int Sa) { return Sa <= 32 ? 1 : (Sa <= 64 ? 2 : (Sa <= 128 ? 4 : 8)); }
template <int RNG>
static const void* event_fn_p(int policy, int R) {
    switch (policy) {
    case MLB_POLICY_SED: return event_fn_r<MLB_POLICY_SED, RNG>(R);
    case MLB_POLICY_LSQ: return event_fn_r<MLB_POLICY_LSQ, RNG>(R);
    case MLB_POLICY_SED2: return event_fn_r<MLB_POLICY_SED2, RNG>(R);
    case MLB_POLICY_LSQ2: return event_fn_r<MLB_POLICY_LSQ2, RNG>(R);
    default: return event_fn_r<MLB_POLICY_ALIAS, RNG>(R);
    }
}
static const void* event_fn(int policy, int Sa, int rng) {
    const int R = lanes_r(Sa);
    return rng == MLB_RNG_PHILOX ? event_fn_p<MLB_RNG_PHILOX>(policy, R) : event_fn_p<MLB_RNG_REPLAY>(policy, R);
}
static const void* feature_fn(int Sa, bool small) {
    switch (lanes_r(Sa)) {
    case 1: return small ? (const void*)feature_kernel<1, true> : (const void*)feature_kernel<1, false>;
    case 2: return small ? (const void*)feature_kernel<2, true> : (const void*)feature_kernel<2, false>;
    case 4: return small ? (const void*)feature_kernel<4, true> : (const void*)feature_kernel<4, false>;
    default: return small ? (const void*)feature_kernel<8, true> : (const void*)feature_kernel<8, false>;
    }
}

template <int CLS>
static const void* pair_fn_c(int Sa) {
    switch (lanes_r(Sa)) {
    case 1: return (const void*)pair_kernel<1, CLS>;
    case 2: return (const void*)pair_kernel<2, CLS>;
    case 4: return (const void*)pair_kernel<4, CLS>;
    default: return (const void*)pair_kernel<8, CLS>;
    }
}

// dynamic shared memory + carve-out sized for `warps_wanted` resident warps (the rest stays L1)
static cudaError_t set_smem(const void* fn, size_t block_bytes, int threads, int warps_wanted) {
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)block_bytes);
    if (e != cudaSuccess) return e;
    const int wpb = threads / 32;
    const int blocks_wanted = wpb >= warps_wanted ? 1 : warps_wanted / wpb;
    const size_t want = (size_t)blocks_wanted * (block_bytes + 1024);
    int pct = (int)((want * 100 + 228 * 1024 - 1) / (228 * 1024));
    pct = pct > 100 ? 100 : pct;
    return cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
}

static int launch_cfg(mlb_env* h) {
    const mlb_config& c = h->cfg;
    const int A = c.num_agents, Sa = c.servers_per_agent;
    const int SP = 32 * lanes_r(Sa);
    const bool alias = c.policy == MLB_POLICY_ALIAS;
    h->ev_threads = 128;
    h->ev_smem = (size_t)(h->ev_threads / 32) * event_warp_smem_bytes(SP, alias);
    h->epb = A == 1 ? 4 : (A == 2 ? 2 : 1);
    h->ft_threads = 32 * A * h->epb;
    h->ft_smem = (size_t)(h->ft_threads / 32) * feature_warp_smem_bytes(SP) + (size_t)h->epb * 2 * h->d.S * 4;
    if (h->ft_threads > 1024) return fail(h, MLB_EINVAL, "num_agents > 32 not supported");
    if (h->ft_smem > 227 * 1024 || h->ev_smem > 227 * 1024)
        return fail(h, MLB_EINVAL, "configuration needs %zu B of shared memory per block (> 227 KB)",
                    h->ft_smem > h->ev_smem ? h->ft_smem : h->ev_smem);
    h->ev_fn = event_fn(c.policy, Sa, c.rng_mode);
    h->ft_fn = feature_fn(Sa, h->ft_threads <= 128);
    cudaError_t e = set_smem(h->ev_fn, h->ev_smem, h->ev_threads, 4 * EV_MIN_BLOCKS);
    if (e == cudaSuccess) e = set_smem(h->ft_fn, h->ft_smem, h->ft_threads, h->ft_threads <= 128 ? 48 : 32);
    h->use_pair = h->d.KP == 128 && c.feature_cache == 1;
    h->d.use_pair = h->use_pair ? 1 : 0;
    h->d.pair_wpe = 1;
    h->pr_smem = (size_t)4 * pair_warp_smem_bytes(SP);
    if (h->use_pair) {
        h->pr_fn[0] = pair_fn_c<0>(Sa);
        h->pr_fn[1] = pair_fn_c<1>(Sa);
        h->pr_fn[2] = pair_fn_c<2>(Sa);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->pair_stream, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->pair_fork, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->pair_join, cudaEventDisableTiming);
        for (int k = 0; k < 3 && e == cudaSuccess; k++) e = set_smem(h->pr_fn[k], h->pr_smem, 128, 32);
    }
    if (e != cudaSuccess) return fail(h, MLB_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    return MLB_OK;
}

static size_t action_elem(int kind) { return kind == MLB_ACTION_DISCRETE_U8 ? 1 : 4; }

// ------------------------------------------------------------------ C ABI
extern "C" {

int mlb_abi_version(void) { return MLB_ABI_VERSION; }

int mlb_config_default(mlb_config* c) {
    if (!c) return MLB_EINVAL;
    memset(c, 0, sizeof *c);
    c->abi_version = MLB_ABI_VERSION;
    c->device = 0;
    c->num_envs = 1;
    c->num_agents = 1;
    c->servers_per_agent = 4;             // env.py:73
    c->reservoir_k = 128;                 // reservoir.py:31
    c->queue_cap = 160;                   // paper 4.2: 32 workers + 128 backlog
    c->policy = MLB_POLICY_SED;
    c->action_kind = MLB_ACTION_DISCRETE_I32;
    c->n_discrete = 3;                    // env.py:69
    c->discrete_weights[0] = 1.0f;
    c->discrete_weights[1] = 1.5f;
    c->discrete_weights[2] = 2.0f;
    c->min_weight = 0.1f;                 // env.py:77
    c->max_weight = 10.0f;                // env.py:76
    c->dt = 0.25f;                        // env.py:80
    c->decay = 0.9;                       // reservoir.py:106
    c->reward_metric = MLB_REWARD_JAIN;   // env.py:78
    c->reward_field = 10;                 // 'flow_duration_avg_decay', env.py:79,380
    c->max_steps = 10000;                 // env.py:81
    c->rng_seed_base = 0;
    c->rng_table_len = 0;
    c->feature_cache = 1;
    c->record_assign = 0;
    return MLB_OK;
}

const char* mlb_last_error(const mlb_env* h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int64_t mlb_launch_count(const mlb_env* h) { return h ? h->launches : 0; }

int mlb_profile_begin(mlb_env* h, int max_steps) {
    if (!h || max_steps < 0) return MLB_EINVAL;
    CK(h, cudaSetDevice(h->device));
    while ((int)h->prof_ev.size() < 4 * max_steps) {
        cudaEvent_t e;
        CK(h, cudaEventCreate(&e));
        h->prof_ev.push_back(e);
    }
    h->prof_cap = max_steps;
    h->prof_n = 0;
    return MLB_OK;
}

int mlb_profile_end(mlb_env* h, double* event_ms, double* feature_ms, int* steps) {
    if (!h) return MLB_EINVAL;
    CK(h, cudaSetDevice(h->device));
    double ev = 0.0, ft = 0.0, pair = 0.0;
    for (int i = 0; i < h->prof_n; i++) {
        float a = 0.f, b = 0.f, c = 0.f;
        CK(h, cudaEventSynchronize(h->prof_ev[(size_t)4 * i + 3]));
        CK(h, cudaEventElapsedTime(&a, h->prof_ev[(size_t)4 * i], h->prof_ev[(size_t)4 * i + 1]));
        CK(h, cudaEventElapsedTime(&c, h->prof_ev[(size_t)4 * i + 1], h->prof_ev[(size_t)4 * i + 2]));
        CK(h, cudaEventElapsedTime(&b, h->prof_ev[(size_t)4 * i + 1], h->prof_ev[(size_t)4 * i + 3]));
        pair += c;
        ev += a;
        ft += b;
    }
    if (event_ms) *event_ms = ev;
    if (feature_ms) *feature_ms = ft;       // statistics pass = pair_kernel + feature_kernel
    h->prof_pair_ms = pair;
    if (steps) *steps = h->prof_n;
    h->prof_cap = 0;
    h->prof_n = 0;
    return MLB_OK;
}

int mlb_destroy(mlb_env* h) {
    if (!h) return MLB_OK;
    cudaSetDevice(h->device);
    for (void* p : h->allocs) cudaFree(p);
    for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
    for (cudaEvent_t e : h->chunk_ev) cudaEventDestroy(e);
    if (h->copy_done) cudaEventDestroy(h->copy_done);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->pair_fork) cudaEventDestroy(h->pair_fork);
    if (h->pair_join) cudaEventDestroy(h->pair_join);
    if (h->pair_stream) cudaStreamDestroy(h->pair_stream);
    delete h->pool;
    for (cudaEvent_t e : h->cr_ev_cnt) cudaEventDestroy(e);
    for (cudaEvent_t e : h->cr_ev_copy) cudaEventDestroy(e);
    if (h->cr_h_rec) cudaFreeHost(h->cr_h_rec);
    if (h->cr_h_col) cudaFreeHost(h->cr_h_col);
    if (h->cr_h_cnt) cudaFreeHost(h->cr_h_cnt);
    if (h->stg_ready) cudaEventDestroy(h->stg_ready);
    if (h->stg_free) cudaEventDestroy(h->stg_free);
    delete h;
    return MLB_OK;
}

int mlb_create(const mlb_config* cfg, mlb_env** out) {
    if (!cfg || !out) return fail(nullptr, MLB_EINVAL, "null argument");
    *out = nullptr;
    const mlb_config& c = *cfg;
    if (c.abi_version != MLB_ABI_VERSION) return fail(nullptr, MLB_EINVAL, "abi_version %d != %d", c.abi_version, MLB_ABI_VERSION);
    if (c.num_envs < 1 || c.num_agents < 1 || c.num_agents > 32) return fail(nullptr, MLB_EINVAL, "num_envs >= 1 and 1 <= num_agents <= 32 required");
    if (c.servers_per_agent < 1 || c.servers_per_agent > 256) return fail(nullptr, MLB_EINVAL, "1 <= servers_per_agent <= 256 required");
    if (c.reservoir_k < 1 || c.reservoir_k > 128) return fail(nullptr, MLB_EINVAL, "1 <= reservoir_k <= 128 required");
    if (c.queue_cap < 1 || c.queue_cap > 65535) return fail(nullptr, MLB_EINVAL, "1 <= queue_cap <= 65535 required");
    if (c.policy < 0 || c.policy > MLB_POLICY_LSQ2) return fail(nullptr, MLB_EINVAL, "unknown policy %d", c.policy);
    if (c.action_kind < 0 || c.action_kind > MLB_ACTION_DISCRETE_U8) return fail(nullptr, MLB_EINVAL, "Unknown action_type: %d", c.action_kind);  // env.py:184
    if (c.action_kind != MLB_ACTION_CONTINUOUS_F32 && (c.n_discrete < 1 || c.n_discrete > 8)) return fail(nullptr, MLB_EINVAL, "1 <= n_discrete <= 8 required");
    if (c.reward_metric < 0 || c.reward_metric >= MLB_REWARD_COUNT_) return fail(nullptr, MLB_EINVAL, "Unsupported metric: %d", c.reward_metric);  // rewards.py:321-323
    if (c.reward_field < 0 || c.reward_field > 10) return fail(nullptr, MLB_EINVAL, "reward_field must be an obs column 0..10");
    if (!(c.dt > 0.f) || !(c.decay > 0.0)) return fail(nullptr, MLB_EINVAL, "dt and decay must be positive");
    if ((double)c.num_envs * c.num_agents * c.servers_per_agent * 2.0 * (((c.reservoir_k + 31) & ~31) / 4) >= 4294967296.0)
        return fail(nullptr, MLB_EINVAL, "num_envs * servers * 2 * K/4 must stay below 2^32 (32-bit reservoir offsets)");
    if ((double)c.num_envs * c.num_agents * c.servers_per_agent * (double)c.queue_cap >= 4294967296.0)
        return fail(nullptr, MLB_EINVAL, "num_envs * servers * queue_cap must stay below 2^32 (32-bit ring offsets)");

    if (c.rng_mode != MLB_RNG_REPLAY && c.rng_mode != MLB_RNG_PHILOX) return fail(nullptr, MLB_EINVAL, "unknown rng_mode %d", c.rng_mode);
    if (c.rng_mode == MLB_RNG_REPLAY &&
        (double)c.num_agents * c.servers_per_agent * (double)(c.rng_table_len > 0 ? c.rng_table_len : 65536) >= 4294967296.0)
        return fail(nullptr, MLB_EINVAL, "servers * rng_table_len must stay below 2^32 (32-bit replay-table offsets)");

    mlb_env* h = new (std::nothrow) mlb_env();
    if (!h) return fail(nullptr, MLB_ENOMEM, "host allocation failed");
    h->cfg = c;
    h->device = c.device;
    auto bail = [&](int code) {
        g_create_err = h->err;
        mlb_destroy(h);
        return code;
    };
#define CKC(call)                                                                   \
    do {                                                                            \
        cudaError_t e__ = (call);                                                   \
        if (e__ != cudaSuccess) {                                                   \
            fail(h, e__ == cudaErrorMemoryAllocation ? MLB_ENOMEM : MLB_ECUDA, "%s failed: %s", #call, cudaGetErrorString(e__)); \
            return bail(e__ == cudaErrorMemoryAllocation ? MLB_ENOMEM : MLB_ECUDA); \
        }                                                                           \
    } while (0)

    CKC(cudaSetDevice(c.device));
    DevState& d = h->d;
    memset(&d, 0, sizeof d);
    d.E = c.num_envs; d.A = c.num_agents; d.Sa = c.servers_per_agent; d.S = d.A * d.Sa;
    d.K = c.reservoir_k; d.KP = (c.reservoir_k + 31) & ~31; d.Q = c.queue_cap;
    d.policy = c.policy; d.action_kind = c.action_kind; d.n_discrete = c.n_discrete;
    d.reward_metric = c.reward_metric; d.reward_field = c.reward_field; d.max_steps = c.max_steps;
    d.L = c.rng_table_len > 0 ? c.rng_table_len : 65536;
    d.feature_cache = c.feature_cache; d.record_assign = c.record_assign;
    d.rng_mode = c.rng_mode; d.rng_key = c.rng_seed_base; d.env_id_base = c.env_id_base;
    for (int i = 0; i < 8; i++) d.dw[i] = c.discrete_weights[i];
    d.min_w = c.min_weight; d.max_w = c.max_weight; d.dt = c.dt;
    d.decay = c.decay; d.log2_decay = (float)std::log2(c.decay);

    const size_t ES = (size_t)d.E * d.S;
    CKC(dalloc(h, &d.n_on, ES));
    CKC(dalloc(h, &d.last_fin, ES));
    CKC(dalloc(h, &d.head, ES));
    CKC(dalloc(h, &d.dropped, ES));
    CKC(dalloc(h, &d.speed, ES));
    CKC(dalloc(h, &d.res_val, ES * 2 * d.KP));
    CKC(dalloc(h, &d.res_ts, ES * 2 * d.KP));
    CKC(dalloc(h, &d.res_count, ES * 2));
    CKC(dalloc(h, &d.res_cursor, ES * 2));
    CKC(dalloc(h, &d.res_rank, ES * 2 * d.KP));
    CKC(dalloc(h, &d.res_chg, ES * 2));
    CKC(dalloc(h, &d.res_tie, ES * 2));
    CKC(dalloc(h, &d.ring, ES * d.Q));
    CKC(dalloc(h, &d.obs, ES * MLB_OBS_COLS));
    CKC(dalloc(h, &d.reward, (size_t)d.E));
    CKC(dalloc(h, &d.done, (size_t)d.E));
    CKC(dalloc(h, &d.step, (size_t)d.E));
    CKC(dalloc(h, &d.arr_cur, (size_t)d.E * d.A));
    CKC(dalloc(h, &d.status, (size_t)1));
    CKC(dalloc(h, &h->d_mask, (size_t)d.E));
    h->action_bytes = ES * action_elem(c.action_kind);
    CKC(dalloc(h, reinterpret_cast<uint8_t**>(&h->d_action), h->action_bytes));
    CKC(cudaMemset(d.status, 0, sizeof(int)));

    // RNG replay table: row j = raw MT19937 words of RandomState(seed_base + j); none in philox mode
    if (c.rng_mode == MLB_RNG_REPLAY) {
        std::vector<uint32_t> tab((size_t)d.S * d.L);
        for (int j = 0; j < d.S; j++) {
            MT19937 g(c.rng_seed_base + (uint32_t)j);
            uint32_t* row = tab.data() + (size_t)j * d.L;
            for (int i = 0; i < d.L; i++) row[i] = g.next();
        }
        uint32_t* t = nullptr;
        CKC(dalloc(h, &t, tab.size()));
        CKC(cudaMemcpy(t, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice));
        d.mt_table = t;
    }
    // SED score table, same arithmetic as the oracle: (float)((double)(n+1) / (1e-9 + (double)w))
    {
        const int TQ = d.Q + 2;
        std::vector<uint32_t> tab((size_t)8 * TQ, 0u);
        for (int a = 0; a < c.n_discrete && a < 8; a++)
            for (int n = 0; n < TQ; n++) {
                const float sc = (float)((double)(n + 1) / (1e-9 + (double)c.discrete_weights[a]));
                uint32_t b;
                memcpy(&b, &sc, 4);
                tab[(size_t)a * TQ + n] = b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);   // = f32_orderable(sc)
            }
        uint32_t* t = nullptr;
        CKC(dalloc(h, &t, tab.size()));
        CKC(cudaMemcpy(t, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice));
        d.sed_table = t;
    }
    // speeds default 1.0
    fill_f32_kernel<<<256, 256>>>(d.speed, ES, 1.0f);
    h->launches++;
    CKC(cudaGetLastError());

    h->state_ptr[MLB_F_N_FLOW_ON] = d.n_on;        h->state_bytes[MLB_F_N_FLOW_ON] = ES * 4;
    h->state_ptr[MLB_F_RES_VALUES] = d.res_val;    h->state_bytes[MLB_F_RES_VALUES] = ES * 2 * d.KP * 4;
    h->state_ptr[MLB_F_RES_TS] = d.res_ts;         h->state_bytes[MLB_F_RES_TS] = ES * 2 * d.KP * 4;
    h->state_ptr[MLB_F_RES_COUNT] = d.res_count;   h->state_bytes[MLB_F_RES_COUNT] = ES * 2 * 4;
    h->state_ptr[MLB_F_RES_CURSOR] = d.res_cursor; h->state_bytes[MLB_F_RES_CURSOR] = ES * 2 * 4;
    h->state_ptr[MLB_F_DROPPED] = d.dropped;       h->state_bytes[MLB_F_DROPPED] = ES * 4;
    h->state_ptr[MLB_F_LAST_FIN] = d.last_fin;     h->state_bytes[MLB_F_LAST_FIN] = ES * 4;
    h->state_ptr[MLB_F_HEAD] = d.head;             h->state_bytes[MLB_F_HEAD] = ES * 4;
    h->state_ptr[MLB_F_STEP] = d.step;             h->state_bytes[MLB_F_STEP] = (size_t)d.E * 4;
    h->state_ptr[MLB_F_OBS] = d.obs;               h->state_bytes[MLB_F_OBS] = ES * MLB_OBS_COLS * 4;
    h->state_ptr[MLB_F_ARR_CURSOR] = d.arr_cur;    h->state_bytes[MLB_F_ARR_CURSOR] = (size_t)d.E * d.A * 4;

    int rc = launch_cfg(h);
    if (rc != MLB_OK) return bail(rc);
    rc = mlb_reset(h, nullptr, nullptr);
    if (rc != MLB_OK) return bail(rc);
    CKC(cudaDeviceSynchronize());
    *out = h;
    return MLB_OK;
#undef CKC
}

int mlb_set_speeds(mlb_env* h, const float* speeds, int64_t n, int loc, void* stream) {
    if (!h || !speeds) return fail(h, MLB_EINVAL, "null argument");
    CK(h, cudaSetDevice(h->device));
    const DevState& d = h->d;
    cudaStream_t st = (cudaStream_t)stream;
    const cudaMemcpyKind kind = loc == MLB_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (n == (int64_t)d.E * d.S) {
        CK(h, cudaMemcpyAsync(d.speed, speeds, (size_t)n * 4, kind, st));
    } else if (n == d.S) {
        std::vector<float> rep;
        if (loc == MLB_HOST) {
            rep.resize((size_t)d.E * d.S);
            for (int e = 0; e < d.E; e++) memcpy(rep.data() + (size_t)e * d.S, speeds, (size_t)d.S * 4);
            CK(h, cudaMemcpyAsync(d.speed, rep.data(), rep.size() * 4, cudaMemcpyHostToDevice, st));
            CK(h, cudaStreamSynchronize(st));
        } else {
            bcast_rows_kernel<<<148 * 4, 256, 0, st>>>(d.speed, speeds, d.S, (size_t)d.E * d.S);
            h->launches++;
            CK(h, cudaGetLastError());
        }
    } else {
        return fail(h, MLB_EINVAL, "speeds: n must be S=%d or E*S=%lld", d.S, (long long)d.E * d.S);
    }
    return MLB_OK;
}

// policies that consume a pre-drawn bucket per flow (alias also consumes u)
static inline bool needs_bucket(int policy) {
    return policy == MLB_POLICY_ALIAS || policy == MLB_POLICY_SED2 || policy == MLB_POLICY_LSQ2;
}

static int alloc_arrivals(mlb_env* h, int64_t total, bool alias) {
    DevState& d = h->d;
    if (total > h->arr_total || (alias && !h->arr_bucket)) {
        // grow-only; old buffers stay in the handle's free list
        CK(h, dalloc(h, &h->arr_time, (size_t)total));
        CK(h, dalloc(h, &h->arr_work, (size_t)total));
        if (alias) {
            CK(h, dalloc(h, &h->arr_bucket, (size_t)total));
            CK(h, dalloc(h, &h->arr_u, (size_t)total));
        }
        if (h->cfg.record_assign) {
            int32_t* a = nullptr;
            CK(h, dalloc(h, &a, (size_t)total));
            d.assign = a;
        }
        h->arr_total = total;
    }
    if (!h->arr_off) {
        CK(h, dalloc(h, &h->arr_off, (size_t)d.E * d.A));
        CK(h, dalloc(h, &h->arr_n, (size_t)d.E * d.A));
    }
    d.arr_time = h->arr_time; d.arr_work = h->arr_work;
    d.arr_bucket = h->arr_bucket; d.arr_u = h->arr_u;
    d.arr_off = h->arr_off; d.arr_n = h->arr_n;
    return MLB_OK;
}

int mlb_load_arrivals(mlb_env* h, const float* time, const float* work, const int32_t* bucket,
                      const float* u, const int64_t* offsets, int loc, void* stream) {
    if (!h || !time || !work || !offsets) return fail(h, MLB_EINVAL, "null argument");
    CK(h, cudaSetDevice(h->device));
    DevState& d = h->d;
    const bool alias = needs_bucket(h->cfg.policy);
    if (h->cfg.policy == MLB_POLICY_ALIAS && (!bucket || !u)) return fail(h, MLB_EINVAL, "alias policy needs pre-drawn bucket/u arrays");
    if (alias && !bucket) return fail(h, MLB_EINVAL, "power-of-two policies need a pre-drawn bucket array");
    cudaStream_t st = (cudaStream_t)stream;
    const int EA = d.E * d.A;
    std::vector<int64_t> off(EA + 1);
    if (loc == MLB_DEVICE) {
        CK(h, cudaMemcpy(off.data(), offsets, (size_t)(EA + 1) * 8, cudaMemcpyDeviceToHost));
    } else {
        memcpy(off.data(), offsets, (size_t)(EA + 1) * 8);
    }
    const int64_t total = off[EA];
    h->h_off.assign(off.begin(), off.begin() + EA);
    h->h_n.resize(EA);
    for (int i = 0; i < EA; i++) {
        const int64_t n = off[i + 1] - off[i];
        if (n < 0 || n > 0x7fffffff) return fail(h, MLB_EINVAL, "offsets must be non-decreasing (stream %d)", i);
        h->h_n[i] = (int32_t)n;
    }
    int rc = alloc_arrivals(h, total > 0 ? total : 1, alias);
    if (rc != MLB_OK) return rc;
    const cudaMemcpyKind kind = loc == MLB_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (total > 0) {
        CK(h, cudaMemcpyAsync(h->arr_time, time, (size_t)total * 4, kind, st));
        CK(h, cudaMemcpyAsync(h->arr_work, work, (size_t)total * 4, kind, st));
        if (alias) {
            CK(h, cudaMemcpyAsync(h->arr_bucket, bucket, (size_t)total * 4, kind, st));
            if (u) {
                CK(h, cudaMemcpyAsync(h->arr_u, u, (size_t)total * 4, kind, st));
            } else {
                CK(h, cudaMemsetAsync(h->arr_u, 0, (size_t)total * 4, st));
            }
        }
    }
    CK(h, cudaMemcpyAsync(h->arr_off, h->h_off.data(), (size_t)EA * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(h->arr_n, h->h_n.data(), (size_t)EA * 4, cudaMemcpyHostToDevice, st));
    CK(h, cudaMemsetAsync(d.arr_cur, 0, (size_t)EA * 4, st));
    CK(h, cudaStreamSynchronize(st));  // host staging vectors must outlive the copies
    h->have_arrivals = true;
    return MLB_OK;
}

// ---- streamed traces: the next chunk of arrivals is copied in on a side stream while the envs step
// through the current one; mlb_commit_arrivals swaps the two buffer sets on the stepping stream.
int mlb_stage_arrivals(mlb_env* h, const float* time, const float* work, const int32_t* bucket, const float* u,
                       const int64_t* offsets, void* copy_stream) {
    if (!h || !offsets) return fail(h, MLB_EINVAL, "null argument");
    CK(h, cudaSetDevice(h->device));
    DevState& d = h->d;
    const bool need_b = needs_bucket(h->cfg.policy);
    const bool empty = offsets[d.E * d.A] == 0;       // a chunk past the end of the trace: pointers may be null
    if (!empty && (!time || !work)) return fail(h, MLB_EINVAL, "null argument");
    if (!empty && h->cfg.policy == MLB_POLICY_ALIAS && (!bucket || !u)) return fail(h, MLB_EINVAL, "alias policy needs pre-drawn bucket/u arrays");
    if (!empty && need_b && !bucket) return fail(h, MLB_EINVAL, "power-of-two policies need a pre-drawn bucket array");
    if (h->cfg.record_assign) return fail(h, MLB_EINVAL, "record_assign is not available with streamed arrivals");
    cudaStream_t cs = (cudaStream_t)copy_stream;
    const int EA = d.E * d.A;
    if (!h->stg_ready) {
        CK(h, cudaEventCreateWithFlags(&h->stg_ready, cudaEventDisableTiming));
        CK(h, cudaEventCreateWithFlags(&h->stg_free, cudaEventDisableTiming));
    }
    if (h->stg_pending) CK(h, cudaEventSynchronize(h->stg_ready));   // host staging vectors are about to be rewritten
    h->stg_h_off.assign(offsets, offsets + EA);
    h->stg_h_n.resize(EA);
    for (int i = 0; i < EA; i++) {
        const int64_t n = offsets[i + 1] - offsets[i];
        if (n < 0 || n > 0x7fffffff) return fail(h, MLB_EINVAL, "offsets must be non-decreasing (stream %d)", i);
        h->stg_h_n[i] = (int32_t)n;
    }
    const int64_t total = offsets[EA] > 0 ? offsets[EA] : 1;
    if (total > h->stg_total || (need_b && !h->stg_bucket)) {
        CK(h, dalloc(h, &h->stg_time, (size_t)total));
        CK(h, dalloc(h, &h->stg_work, (size_t)total));
        if (need_b) {
            CK(h, dalloc(h, &h->stg_bucket, (size_t)total));
            CK(h, dalloc(h, &h->stg_u, (size_t)total));
        }
        h->stg_total = total;
    }
    if (!h->stg_off) {
        CK(h, dalloc(h, &h->stg_off, (size_t)EA));
        CK(h, dalloc(h, &h->stg_n, (size_t)EA));
    }
    CK(h, cudaStreamWaitEvent(cs, h->stg_free, 0));   // no-op until the first commit has recorded it
    if (offsets[EA] > 0) {
        const size_t nb = (size_t)offsets[EA] * 4;
        CK(h, cudaMemcpyAsync(h->stg_time, time, nb, cudaMemcpyHostToDevice, cs));
        CK(h, cudaMemcpyAsync(h->stg_work, work, nb, cudaMemcpyHostToDevice, cs));
        if (need_b) {
            CK(h, cudaMemcpyAsync(h->stg_bucket, bucket, nb, cudaMemcpyHostToDevice, cs));
            if (u) {
                CK(h, cudaMemcpyAsync(h->stg_u, u, nb, cudaMemcpyHostToDevice, cs));
            } else {
                CK(h, cudaMemsetAsync(h->stg_u, 0, nb, cs));
            }
        }
    }
    CK(h, cudaMemcpyAsync(h->stg_off, h->stg_h_off.data(), (size_t)EA * 8, cudaMemcpyHostToDevice, cs));
    CK(h, cudaMemcpyAsync(h->stg_n, h->stg_h_n.data(), (size_t)EA * 4, cudaMemcpyHostToDevice, cs));
    CK(h, cudaEventRecord(h->stg_ready, cs));
    h->stg_pending = true;
    h->stg_valid = true;
    return MLB_OK;
}

int mlb_commit_arrivals(mlb_env* h, void* stream) {
    if (!h) return MLB_EINVAL;
    if (!h->stg_valid) return fail(h, MLB_ESTATE, "mlb_commit_arrivals without a staged chunk");
    CK(h, cudaSetDevice(h->device));
    DevState& d = h->d;
    cudaStream_t st = (cudaStream_t)stream;
    CK(h, cudaStreamWaitEvent(st, h->stg_ready, 0));
    CK(h, cudaEventRecord(h->stg_free, st));          // every earlier step on `st` is done with the old chunk by then
    std::swap(h->arr_time, h->stg_time); std::swap(h->arr_work, h->stg_work);
    std::swap(h->arr_bucket, h->stg_bucket); std::swap(h->arr_u, h->stg_u);
    std::swap(h->arr_off, h->stg_off); std::swap(h->arr_n, h->stg_n);
    std::swap(h->arr_total, h->stg_total);
    h->h_off.swap(h->stg_h_off);
    h->h_n.swap(h->stg_h_n);
    d.arr_time = h->arr_time; d.arr_work = h->arr_work;
    d.arr_bucket = h->arr_bucket; d.arr_u = h->arr_u;
    d.arr_off = h->arr_off; d.arr_n = h->arr_n;
    CK(h, cudaMemsetAsync(d.arr_cur, 0, (size_t)d.E * d.A * 4, st));
    h->stg_valid = false;
    h->have_arrivals = true;
    return MLB_OK;
}

int mlb_gen_poisson(mlb_env* h, double rate, double mean_work, double horizon, uint64_t seed, void* stream) {
    return mlb_gen_poisson_window(h, rate, mean_work, 0.0, horizon, seed, 0u, stream);
}

int mlb_gen_poisson_window(mlb_env* h, double rate, double mean_work, double t_start, double t_end, uint64_t seed,
                           uint32_t window, void* stream) {
    if (!h) return MLB_EINVAL;
    const double horizon = t_end;
    if (!(rate > 0) || !(mean_work > 0) || !(t_start >= 0) || !(t_end > t_start))
        return fail(h, MLB_EINVAL, "rate, mean_work must be positive and 0 <= t_start < t_end");
    CK(h, cudaSetDevice(h->device));
    DevState& d = h->d;
    cudaStream_t st = (cudaStream_t)stream;
    const int EA = d.E * d.A;
    const double mu = rate * (t_end - t_start);
    const int cap = (int)(mu + 8.0 * std::sqrt(mu) + 64.0);
    const bool alias = needs_bucket(h->cfg.policy);
    int rc = alloc_arrivals(h, (int64_t)EA * cap, alias);
    if (rc != MLB_OK) return rc;
    h->h_off.resize(EA);
    for (int i = 0; i < EA; i++) h->h_off[i] = (int64_t)i * cap;
    CK(h, cudaMemcpyAsync(h->arr_off, h->h_off.data(), (size_t)EA * 8, cudaMemcpyHostToDevice, st));
    const int threads = 128;
    const int blocks = (int)(((int64_t)EA * 32 + threads - 1) / threads);
    gen_poisson_kernel<<<blocks, threads, 0, st>>>(h->arr_time, h->arr_work, alias ? h->arr_bucket : nullptr,
                                                   alias ? h->arr_u : nullptr, h->arr_n, EA, cap, d.Sa,
                                                   (uint32_t)h->cfg.env_id_base * (uint32_t)d.A,
                                                   rate, mean_work, t_start, horizon, seed, window);
    h->launches++;
    CK(h, cudaGetLastError());
    CK(h, cudaMemsetAsync(d.arr_cur, 0, (size_t)EA * 4, st));
    h->h_n.resize(EA);
    CK(h, cudaMemcpyAsync(h->h_n.data(), h->arr_n, (size_t)EA * 4, cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    h->have_arrivals = true;
    return MLB_OK;
}

int mlb_get_arrivals(mlb_env* h, int32_t env, int32_t agent, float* time, float* work,
                     int32_t* bucket, float* u, int64_t cap, int64_t* n) {
    if (!h || !n) return MLB_EINVAL;
    if (!h->have_arrivals) return fail(h, MLB_ESTATE, "no arrivals loaded");
    const DevState& d = h->d;
    if (env < 0 || env >= d.E || agent < 0 || agent >= d.A) return fail(h, MLB_EINVAL, "env/agent out of range");
    CK(h, cudaSetDevice(h->device));
    const int ea = env * d.A + agent;
    const int64_t cnt = h->h_n[ea], off = h->h_off[ea];
    *n = cnt;
    const int64_t m = cnt < cap ? cnt : cap;
    if (m > 0) {
        if (time) CK(h, cudaMemcpy(time, h->arr_time + off, (size_t)m * 4, cudaMemcpyDeviceToHost));
        if (work) CK(h, cudaMemcpy(work, h->arr_work + off, (size_t)m * 4, cudaMemcpyDeviceToHost));
        if (bucket && h->arr_bucket) CK(h, cudaMemcpy(bucket, h->arr_bucket + off, (size_t)m * 4, cudaMemcpyDeviceToHost));
        if (u && h->arr_u) CK(h, cudaMemcpy(u, h->arr_u + off, (size_t)m * 4, cudaMemcpyDeviceToHost));
    }
    return MLB_OK;
}

int mlb_reset(mlb_env* h, const uint8_t* env_mask, void* stream) {
    if (!h) return MLB_EINVAL;
    CK(h, cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const uint8_t* dm = nullptr;
    if (env_mask) {
        CK(h, cudaMemcpyAsync(h->d_mask, env_mask, (size_t)h->d.E, cudaMemcpyHostToDevice, st));
        dm = h->d_mask;
    }
    reset_kernel<<<h->d.E, 256, 0, st>>>(h->d, dm);
    h->launches++;
    CK(h, cudaGetLastError());
    return MLB_OK;
}

// the two kernels of one env step over envs [e0, e1)
static int launch_step(mlb_env* h, const void* dact, int e0, int e1, cudaStream_t st, cudaEvent_t* pe) {
    DevState dv = h->d;
    dv.e0 = e0;
    dv.e1 = e1;
    const void* act = dact;
    void* ev_args[] = {&dv, &act};
    const int wpb = h->ev_threads / 32;
    const int ev_blocks = (int)(((int64_t)(e1 - e0) * dv.A + wpb - 1) / wpb);
    if (pe) CK(h, cudaEventRecord(pe[0], st));
    CK(h, cudaLaunchKernel(h->ev_fn, dim3(ev_blocks), dim3(h->ev_threads), ev_args, h->ev_smem, st));
    if (pe) CK(h, cudaEventRecord(pe[1], st));
    void* ft_args[] = {&dv};
    if (h->use_pair) {
        const int64_t pairs = (int64_t)(e1 - e0) * dv.A;
        if (pairs <= 8192) {
            // four warps per (env, agent), both classes side by side
            dv.pair_wpe = 4;
            CK(h, cudaEventRecord(h->pair_fork, st));
            CK(h, cudaStreamWaitEvent(h->pair_stream, h->pair_fork, 0));
            CK(h, cudaLaunchKernel(h->pr_fn[0], dim3((int)pairs), dim3(128), ft_args, h->pr_smem, st));
            CK(h, cudaLaunchKernel(h->pr_fn[1], dim3((int)pairs), dim3(128), ft_args, h->pr_smem, h->pair_stream));
            CK(h, cudaEventRecord(h->pair_join, h->pair_stream));
            CK(h, cudaStreamWaitEvent(st, h->pair_join, 0));
            h->launches += 2;
        } else {
            // one warp per (env, agent), both classes in one launch
            CK(h, cudaLaunchKernel(h->pr_fn[2], dim3((int)((pairs + 3) / 4)), dim3(128), ft_args, h->pr_smem, st));
            h->launches += 1;
        }
    }
    if (pe) CK(h, cudaEventRecord(pe[2], st));
    const int ft_blocks = (e1 - e0 + h->epb - 1) / h->epb;
    CK(h, cudaLaunchKernel(h->ft_fn, dim3(ft_blocks), dim3(h->ft_threads), ft_args, h->ft_smem, st));
    if (pe) CK(h, cudaEventRecord(pe[3], st));
    h->launches += 2;
    return MLB_OK;
}

int mlb_step(mlb_env* h, const void* action, int action_loc, float* out_obs, double* out_reward,
             uint8_t* out_done, int out_loc, void* stream) {
    if (!h || !action) return fail(h, MLB_EINVAL, "null argument");
    if (!h->have_arrivals) return fail(h, MLB_ESTATE, "mlb_step before mlb_load_arrivals / mlb_gen_poisson");
    CK(h, cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const DevState& d = h->d;
    const size_t S = (size_t)d.S;
    const size_t asz = action_elem(d.action_kind);

    // ---- host buffers on both sides and enough envs: pipeline the step in chunks of envs, so
    // that the device->host copy of chunk c's observations (the bulk of the bytes) overlaps the
    // kernels of chunk c+1.  Envs are independent, so any split gives the same result.
    const int n_chunks = h->host_chunks;
    if (action_loc == MLB_HOST && out_loc == MLB_HOST && out_obs && n_chunks > 1 && d.E >= n_chunks * 1024) {
        if (!h->copy_stream) {
            CK(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
            CK(h, cudaEventCreateWithFlags(&h->copy_done, cudaEventDisableTiming));
        }
        while ((int)h->chunk_ev.size() < n_chunks) {
            cudaEvent_t e;
            CK(h, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            h->chunk_ev.push_back(e);
        }
        const int per = ((d.E + n_chunks - 1) / n_chunks + h->epb - 1) / h->epb * h->epb;
        int c = 0;
        for (int e0 = 0; e0 < d.E; e0 += per, c++) {
            const int e1 = e0 + per < d.E ? e0 + per : d.E;
            const size_t ne = (size_t)(e1 - e0);
            CK(h, cudaMemcpyAsync((char*)h->d_action + (size_t)e0 * S * asz, (const char*)action + (size_t)e0 * S * asz,
                                  ne * S * asz, cudaMemcpyHostToDevice, st));
            const int rc = launch_step(h, h->d_action, e0, e1, st, nullptr);
            if (rc != MLB_OK) return rc;
            CK(h, cudaEventRecord(h->chunk_ev[c], st));
            CK(h, cudaStreamWaitEvent(h->copy_stream, h->chunk_ev[c], 0));
            CK(h, cudaMemcpyAsync(out_obs + (size_t)e0 * S * MLB_OBS_COLS, d.obs + (size_t)e0 * S * MLB_OBS_COLS,
                                  ne * S * MLB_OBS_COLS * 4, cudaMemcpyDeviceToHost, h->copy_stream));
        }
        CK(h, cudaGetLastError());
        if (out_reward) CK(h, cudaMemcpyAsync(out_reward, d.reward, (size_t)d.E * 8, cudaMemcpyDeviceToHost, st));
        if (out_done) CK(h, cudaMemcpyAsync(out_done, d.done, (size_t)d.E, cudaMemcpyDeviceToHost, st));
        CK(h, cudaEventRecord(h->copy_done, h->copy_stream));
        CK(h, cudaStreamWaitEvent(st, h->copy_done, 0));  // the caller's stream covers the copies too
        return MLB_OK;
    }

    const void* dact = action;
    if (action_loc == MLB_HOST) {
        CK(h, cudaMemcpyAsync(h->d_action, action, h->action_bytes, cudaMemcpyHostToDevice, st));
        dact = h->d_action;
    }
    const bool prof = h->prof_n < h->prof_cap;
    {
        const int rc = launch_step(h, dact, 0, d.E, st, prof ? &h->prof_ev[(size_t)4 * h->prof_n] : nullptr);
        if (rc != MLB_OK) return rc;
        if (prof) h->prof_n++;
    }
    CK(h, cudaGetLastError());
    const cudaMemcpyKind kind = out_loc == MLB_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    const size_t ES = (size_t)d.E * d.S;
    if (out_obs) CK(h, cudaMemcpyAsync(out_obs, d.obs, ES * MLB_OBS_COLS * 4, kind, st));
    if (out_reward) CK(h, cudaMemcpyAsync(out_reward, d.reward, (size_t)d.E * 8, kind, st));
    if (out_done) CK(h, cudaMemcpyAsync(out_done, d.done, (size_t)d.E, kind, st));
    return MLB_OK;
}

// End-to-end step that moves only what changed (see the header).  Synchronous.
int mlb_step_changed(mlb_env* h, const void* action, float* host_obs, double* out_reward, uint8_t* out_done,
                     int threads, int64_t* d2h_bytes, void* stream) {
    if (!h || !action || !host_obs) return fail(h, MLB_EINVAL, "null argument");
    if (!h->have_arrivals) return fail(h, MLB_ESTATE, "mlb_step before mlb_load_arrivals / mlb_gen_poisson");
    CK(h, cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const DevState& d = h->d;
    const size_t S = (size_t)d.S, ES = (size_t)d.E * S;
    const size_t asz = action_elem(d.action_kind);
    int n_chunks = d.E >= h->host_chunks * 1024 ? h->host_chunks : 1;
    if (n_chunks < 1) n_chunks = 1;
    if (!h->cr_rec) {
        CK(h, dalloc(h, &h->cr_rec, ES * 12));
        CK(h, dalloc(h, &h->cr_col, ES));
        CK(h, dalloc(h, &h->cr_cnt, (size_t)64));
        CK(h, cudaMallocHost((void**)&h->cr_h_rec, ES * 48));
        CK(h, cudaMallocHost((void**)&h->cr_h_col, ES * 2));
        CK(h, cudaMallocHost((void**)&h->cr_h_cnt, 64 * 4));
    }
    if (n_chunks > 64) n_chunks = 64;
    if (!h->copy_stream) {
        CK(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        CK(h, cudaEventCreateWithFlags(&h->copy_done, cudaEventDisableTiming));
    }
    while ((int)h->cr_ev_cnt.size() < n_chunks) {
        cudaEvent_t a, b;
        CK(h, cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
        CK(h, cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
        h->cr_ev_cnt.push_back(a);
        h->cr_ev_copy.push_back(b);
    }
    if (threads <= 0) {
        threads = (int)std::thread::hardware_concurrency();
        threads = threads > 16 ? 16 : (threads < 1 ? 1 : threads);
    }
    if (!h->pool || (int)h->pool->th.size() != threads) {
        delete h->pool;
        h->pool = new HostPool(threads);
    }
    const int per = ((d.E + n_chunks - 1) / n_chunks + h->epb - 1) / h->epb * h->epb;
    // ---- phase 1: every chunk's kernels, compaction and record count, back to back on the caller's stream
    CK(h, cudaMemsetAsync(h->cr_cnt, 0, 64 * 4, st));
    int nc = 0;
    for (int e0 = 0; e0 < d.E; e0 += per, nc++) {
        const int e1 = e0 + per < d.E ? e0 + per : d.E;
        const size_t ne = (size_t)(e1 - e0);
        CK(h, cudaMemcpyAsync((char*)h->d_action + (size_t)e0 * S * asz, (const char*)action + (size_t)e0 * S * asz,
                              ne * S * asz, cudaMemcpyHostToDevice, st));
        const int rc = launch_step(h, h->d_action, e0, e1, st, nullptr);
        if (rc != MLB_OK) return rc;
        DevState dv = h->d;
        dv.e0 = e0;
        dv.e1 = e1;
        const size_t rows = ne * S;
        compact_rows_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(dv, h->cr_rec, h->cr_col, h->cr_cnt + nc);
        h->launches++;
        CK(h, cudaMemcpyAsync(h->cr_h_cnt + nc, h->cr_cnt + nc, 4, cudaMemcpyDeviceToHost, st));
        CK(h, cudaEventRecord(h->cr_ev_cnt[nc], st));
    }
    CK(h, cudaGetLastError());
    if (out_reward) CK(h, cudaMemcpyAsync(out_reward, d.reward, (size_t)d.E * 8, cudaMemcpyDeviceToHost, st));
    if (out_done) CK(h, cudaMemcpyAsync(out_done, d.done, (size_t)d.E, cudaMemcpyDeviceToHost, st));
    // ---- phase 2: per chunk, as soon as its count is known: the records + the n_flow_on column (or, when most rows
    // changed, the chunk's observation block straight into place) on the copy stream; the host threads apply chunk
    // c - 1 while chunk c is on the wire
    int64_t moved = 0;
    std::vector<uint32_t> n_rec(nc);
    std::vector<char> sparse(nc);
    auto apply = [&](int c) -> int {
        CK(h, cudaEventSynchronize(h->cr_ev_copy[c]));
        if (!sparse[c]) return MLB_OK;
        const int e0 = c * per, e1 = e0 + per < d.E ? e0 + per : d.E;
        const size_t row0 = (size_t)e0 * S, rows = (size_t)(e1 - e0) * S;
        const uint32_t* rec = h->cr_h_rec + row0 * 12;
        const uint16_t* col = h->cr_h_col + row0;
        const uint32_t n = n_rec[c];
        h->pool->run([=](int t, int nt) {
            const size_t a = rows * (size_t)t / nt, b = rows * (size_t)(t + 1) / nt;
            for (size_t i = a; i < b; i++) {                     // n_flow_on of every row; untouched lines stay clean
                float* o = host_obs + (row0 + i) * MLB_OBS_COLS;
                const float v = (float)col[i];
                if (*o != v) *o = v;
            }
            const size_t ra = (size_t)n * t / nt, rb = (size_t)n * (t + 1) / nt;
            for (size_t k = ra; k < rb; k++) {
                const uint32_t* r = rec + k * 12;
                memcpy(host_obs + (size_t)r[0] * MLB_OBS_COLS, r + 1, MLB_OBS_COLS * 4);
            }
        });
        return MLB_OK;
    };
    for (int c = 0; c < nc; c++) {
        const int e0 = c * per, e1 = e0 + per < d.E ? e0 + per : d.E;
        const size_t row0 = (size_t)e0 * S, rows = (size_t)(e1 - e0) * S;
        CK(h, cudaEventSynchronize(h->cr_ev_cnt[c]));
        const uint32_t n = h->cr_h_cnt[c];
        n_rec[c] = n;
        sparse[c] = (size_t)n * 48 + rows * 2 < rows * MLB_OBS_COLS * 4 * 3 / 4;
        if (sparse[c]) {
            CK(h, cudaMemcpyAsync(h->cr_h_col + row0, h->cr_col + row0, rows * 2, cudaMemcpyDeviceToHost, h->copy_stream));
            if (n) CK(h, cudaMemcpyAsync(h->cr_h_rec + row0 * 12, h->cr_rec + row0 * 12, (size_t)n * 48, cudaMemcpyDeviceToHost, h->copy_stream));
            moved += (int64_t)rows * 2 + (int64_t)n * 48 + 4;
        } else {
            CK(h, cudaMemcpyAsync(host_obs + row0 * MLB_OBS_COLS, d.obs + row0 * MLB_OBS_COLS, rows * MLB_OBS_COLS * 4,
                                  cudaMemcpyDeviceToHost, h->copy_stream));
            moved += (int64_t)rows * MLB_OBS_COLS * 4 + 4;
        }
        CK(h, cudaEventRecord(h->cr_ev_copy[c], h->copy_stream));
        if (c > 0) {
            const int rc = apply(c - 1);
            if (rc != MLB_OK) return rc;
        }
    }
    {
        const int rc = apply(nc - 1);
        if (rc != MLB_OK) return rc;
    }
    CK(h, cudaStreamSynchronize(st));
    if (d2h_bytes) *d2h_bytes = moved + (out_reward ? (int64_t)d.E * 8 : 0) + (out_done ? (int64_t)d.E : 0);
    return MLB_OK;
}

double mlb_profile_pair_ms(const mlb_env* h) { return h ? h->prof_pair_ms : 0.0; }

int mlb_get_assignments(mlb_env* h, int32_t* dst, int64_t n, int loc, void* stream) {
    if (!h || !dst) return MLB_EINVAL;
    if (!h->d.assign) return fail(h, MLB_ESTATE, "record_assign was not enabled");
    if (n > h->arr_total) return fail(h, MLB_EINVAL, "n exceeds the number of loaded flows");
    CK(h, cudaSetDevice(h->device));
    CK(h, cudaMemcpyAsync(dst, h->d.assign, (size_t)n * 4,
                          loc == MLB_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost,
                          (cudaStream_t)stream));
    if (loc == MLB_HOST) CK(h, cudaStreamSynchronize((cudaStream_t)stream));
    return MLB_OK;
}

int mlb_device_ptr(mlb_env* h, int what, void** ptr, size_t* bytes) {
    if (!h || !ptr) return MLB_EINVAL;
    const DevState& d = h->d;
    size_t b = 0;
    void* p = nullptr;
    if (what >= 0 && what < MLB_F_COUNT_) { p = h->state_ptr[what]; b = h->state_bytes[what]; }
    else if (what == MLB_PTR_OBS) { p = d.obs; b = (size_t)d.E * d.S * MLB_OBS_COLS * 4; }
    else if (what == MLB_PTR_REWARD) { p = d.reward; b = (size_t)d.E * 8; }
    else if (what == MLB_PTR_DONE) { p = d.done; b = (size_t)d.E; }
    else if (what == MLB_PTR_ASSIGN) { p = d.assign; b = (size_t)h->arr_total * 4; }
    else return fail(h, MLB_EINVAL, "unknown pointer id %d", what);
    *ptr = p;
    if (bytes) *bytes = b;
    return MLB_OK;
}

int mlb_get_state(mlb_env* h, int field, void* dst, size_t bytes, int loc) {
    if (!h || !dst) return MLB_EINVAL;
    if (field < 0 || field >= MLB_F_COUNT_) return fail(h, MLB_EINVAL, "unknown field %d", field);
    if (bytes != h->state_bytes[field]) return fail(h, MLB_EINVAL, "field %d is %zu bytes, caller passed %zu", field, h->state_bytes[field], bytes);
    CK(h, cudaSetDevice(h->device));
    CK(h, cudaDeviceSynchronize());
    CK(h, cudaMemcpy(dst, h->state_ptr[field], bytes, loc == MLB_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost));
    return MLB_OK;
}

int mlb_status(mlb_env* h, void* stream) {
    if (!h) return MLB_EINVAL;
    CK(h, cudaSetDevice(h->device));
    int st = 0;
    CK(h, cudaMemcpyAsync(&st, h->d.status, sizeof st, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CK(h, cudaStreamSynchronize((cudaStream_t)stream));
    if (st & ST_ERR_RNG) return fail(h, MLB_ERNG, "replayed MT19937 stream exhausted: raise rng_table_len (now %d words per seed)", h->d.L);
    if (st & ST_ERR_ACTION) return fail(h, MLB_EACTION, "discrete action outside [0, %d)", h->d.n_discrete);
    return MLB_OK;
}

int mlb_mt19937_fill(uint32_t seed, uint32_t* out, int64_t n) {
    if (!out || n < 0) return MLB_EINVAL;
    MT19937 g(seed);
    for (int64_t i = 0; i < n; i++) out[i] = g.next();
    return MLB_OK;
}

}  // extern "C"
