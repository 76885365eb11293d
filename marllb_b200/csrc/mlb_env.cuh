// Device-side state description shared by the env kernels and the C ABI.
#pragma once
#include <stdint.h>

namespace mlb {

enum : int { ST_ERR_RNG = 1, ST_ERR_ACTION = 2 };

// Everything a kernel needs, passed by value (fits the 4 KB param space).
struct DevState {
    // ---- configuration
    int E, A, Sa, S;       // envs, agents/env, servers/agent, S = A*Sa
    int e0, e1;            // env range [e0, e1) of this launch (host-buffer steps are pipelined in chunks)
    int K, KP, Q;          // reservoir capacity, padded stride (mult. of 32), queue cap
    int policy, action_kind, n_discrete;
    int reward_metric, reward_field, max_steps;
    int L;                 // words per MT19937 replay row
    int feature_cache, record_assign;
    int use_pair;          // pair_kernel evaluates the "fast" reservoirs before feature_kernel
    int pair_wpe;          // warps per (env, agent) in pair_kernel: 1, or 4 (small launches: the list is dealt out to a block)
    int rng_mode;          // MLB_RNG_REPLAY (table rows of RandomState(seed_base + j)) or MLB_RNG_PHILOX (per env)
    uint32_t rng_key;      // philox mode: key word 0 (= rng_seed_base)
    int env_id_base;       // global id of env 0 (philox streams are keyed by the GLOBAL env id)
    float dw[8];
    float min_w, max_w, dt;
    float log2_decay;
    double decay;
    // ---- per-server state, SoA over [E][S]
    int32_t* n_on;         // n_flow_on                      (src/vpp/lb/shm.h:31-33)
    float* last_fin;       // finish time of the newest queued flow
    uint32_t* head;        // ring position of the oldest in-system flow
    uint32_t* dropped;
    float* speed;
    // ---- reservoirs: [E][S][2][KP] values/timestamps, [E][2][S] counters
    float* res_val;
    float* res_ts;
    uint32_t* res_count;
    uint32_t* res_cursor;
    uint8_t* res_rank;     // [E][S][2][KP] rank of each slot's value (order statistics cache)
    uint32_t* res_chg;     // [E][2][S] slots written this step (event kernel -> feature kernel)
    uint8_t* res_tie;      // [E][2][S] 1: the last p90_decay decision was an exact tie (feature kernel re-evaluates it)
    // ---- FIFO rings [E][S][Q]
    float2* ring;          // (arrival time, finish time) of every in-system flow
    // ---- outputs
    float* obs;            // [E][S][11]
    double* reward;        // [E]
    uint8_t* done;         // [E]
    int32_t* step;         // [E]
    // ---- arrivals, one stream per (env, agent)
    const float* arr_time;
    const float* arr_work;
    const int32_t* arr_bucket;
    const float* arr_u;
    const int64_t* arr_off; // [E*A]
    const int32_t* arr_n;   // [E*A]
    int32_t* arr_cur;       // [E*A]
    int32_t* assign;        // parallel to arr_time (optional)
    // ---- RNG replay table [S][L] and sticky status word
    const uint32_t* mt_table;
    const uint32_t* sed_table; // [n_discrete][Q+2] SED scores for discrete actions as order-preserving uints (host-built)
    int* status;
};

}  // namespace mlb
