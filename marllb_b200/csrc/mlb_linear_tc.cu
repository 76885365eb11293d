// y = act(x W^T + b) on the 5th-generation tensor cores (tcgen05, sm_100a), fp32 in / fp32 out.
//
// The dense contractions of the batched policy forward (reference: nn.GRU / nn.Linear inside
// simulation-mode/problem-05-qmix/src/agent_network.py:63-87 and
// simulation-mode/problem-04-sac-gru/src/networks.py:82-147, 209-237) at rollout batch sizes
// (M = envs x agents in the thousands).  The parity bar is 1e-5 relative against the fp32
// reference, which a single TF32 product (10-bit mantissa) cannot meet, so every operand is
// split in the kernel into a TF32 "hi" part and a TF32 "lo" remainder and three MMAs are
// accumulated in fp32 in tensor memory (3xTF32):  x.w ~= xh.wh + xh.wl + xl.wh.
// The tensor core rounds its fp32 accumulator toward zero on every instruction (measured: the
// error of a single long accumulation grows linearly with K, 2e-5 relative at K = 2816), so the
// accumulator in tensor memory only ever holds ONE 32-wide k-block: the worker warps drain it
// into per-thread fp32 registers (round-to-nearest adds) while the next k-block is being
// multiplied into the other half of a double-buffered accumulator.
//
// One CTA = one 128 x NT output tile (NT = 32 / 64 / 128), 10 warps:
//   warp 0      TMA producer: x tile [128 x 32] and W tile [NT x 32] (fp32, 128-byte swizzle)
//   warp 1      allocates tensor memory, issues tcgen05.mma (one elected lane), frees it
//   warps 2..9  split hi/lo in shared memory (in place + a second buffer with the same swizzled
//               addresses), drain the previous k-block's partial sums (tcgen05.ld: warp w owns TMEM
//               lanes 32(w%4).., half of the columns), then the epilogue from registers
// Shared memory: a 4-deep TMA ring of raw tiles (covers the DRAM latency) and a 2-deep ring of "lo"
// tiles.  mbarriers: full (TMA -> split), ready (split -> MMA), raw_empty / lo_empty
// (tcgen05.commit -> TMA / split), pfull (tcgen05.commit -> drain), drained (drain -> MMA).
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/marllb_b200.h"
#include "../../include/marllb_b200_policy.h"
#include "mlb_tc_common.cuh"

namespace {
using namespace mlb_tc;

constexpr int LO_STAGES = 2;        // ring of the "lo" remainders computed by the worker warps
constexpr int DRAIN_KB = 2;         // k-blocks accumulated in tensor memory before the partial sums are drained
// RAW_STAGES (template): TMA ring of raw fp32 tiles (= the "hi" operands: the MMA ignores the low 13 bits)
constexpr int WORKER_WARPS = 8;
constexpr int SPLIT_THREADS = 32 * WORKER_WARPS;   // 256
constexpr int THREADS = 64 + SPLIT_THREADS;        // + TMA warp + MMA warp

struct TcParams {
    float* C;
    const float* bias;
    int64_t ldc;
    int M, N, K, act;
    int tma_store;   // C goes out through shared memory + TMA (coalesced, clipped at the matrix edge)
};

__device__ __forceinline__ float apply_act(float v, int act) {
    if (act == MLB_ACT_RELU) return fmaxf(v, 0.f);
    if (act == MLB_ACT_ABS) return fabsf(v);
    return v;
}

template <int NT, int RAW_STAGES>
__global__ void __launch_bounds__(THREADS, 1)
linear_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                 const __grid_constant__ CUtensorMap map_c, const TcParams p) {
    extern __shared__ unsigned char smem_dyn[];
    // 1024-byte alignment for the swizzled tiles
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
    constexpr uint32_t a_bytes = TILE_M * TILE_K * 4;         // 16 KB
    constexpr uint32_t b_bytes = (uint32_t)NT * TILE_K * 4;
    constexpr uint32_t stage_bytes = a_bytes + b_bytes;            // A | B  (raw ring and lo ring alike)
    constexpr uint32_t TMEM_COLS = 2 * NT <= 32 ? 32 : (2 * NT <= 64 ? 64 : (2 * NT <= 128 ? 128 : (2 * NT <= 256 ? 256 : 512)));   // double-buffered partial accumulator
    unsigned char* lo_base = smem + (size_t)RAW_STAGES * stage_bytes;
    unsigned char* bars = lo_base + (size_t)LO_STAGES * stage_bytes;
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto raw_empty_bar = [&](int s) { return bar0 + 8u * (RAW_STAGES + s); };
    auto ready_bar = [&](int s) { return bar0 + 8u * (2 * RAW_STAGES + s); };
    auto lo_empty_bar = [&](int s) { return bar0 + 8u * (2 * RAW_STAGES + LO_STAGES + s); };
    auto pfull_bar = [&](int b) { return bar0 + 8u * (2 * RAW_STAGES + 2 * LO_STAGES + b); };
    auto drained_bar = [&](int b) { return bar0 + 8u * (2 * RAW_STAGES + 2 * LO_STAGES + 2 + b); };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(bars + 8 * (2 * RAW_STAGES + 2 * LO_STAGES + 4));

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int m0 = blockIdx.y * TILE_M;
    const int n0 = blockIdx.x * NT;     // N tiles of one row block are neighbours in launch order: x tile reuse in L2
    const int nkb = (p.K + TILE_K - 1) / TILE_K;

    if (threadIdx.x == 0) {
        for (int s = 0; s < RAW_STAGES; s++) {
            mbar_init(full_bar(s), 1);
            mbar_init(raw_empty_bar(s), 1);
        }
        for (int s = 0; s < LO_STAGES; s++) {
            mbar_init(ready_bar(s), WORKER_WARPS);      // one arrival per worker warp
            mbar_init(lo_empty_bar(s), 1);
        }
        for (int b = 0; b < 2; b++) {
            mbar_init(pfull_bar(b), 1);
            mbar_init(drained_bar(b), WORKER_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)),
                     "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------ TMA producer
        if (elect_one()) {
            for (int kb = 0; kb < nkb; kb++) {
                const int s = kb % RAW_STAGES;
                mbar_wait(raw_empty_bar(s), ((kb / RAW_STAGES) & 1) ^ 1);
                const uint32_t a_hi = smem_u32(smem + (size_t)s * stage_bytes);
                const uint32_t b_hi = a_hi + a_bytes;
                mbar_arrive_expect_tx(full_bar(s), a_bytes + b_bytes);
                tma_load_2d(a_hi, &map_x, kb * TILE_K, m0, full_bar(s));
                tma_load_2d(b_hi, &map_w, kb * TILE_K, n0, full_bar(s));
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------ MMA issuer
        const uint32_t idesc = umma_idesc_tf32(TILE_M, NT);
        for (int kb = 0; kb < nkb; kb++) {
            const int s = kb % RAW_STAGES, sl = kb % LO_STAGES;
            const int ch = kb / DRAIN_KB, pb = ch & 1;
            const bool first = kb % DRAIN_KB == 0, last = kb % DRAIN_KB == DRAIN_KB - 1 || kb == nkb - 1;
            mbar_wait(ready_bar(sl), (kb / LO_STAGES) & 1);    // lo tiles written (and the raw stage landed)
            if (first) mbar_wait(drained_bar(pb), ((ch >> 1) & 1) ^ 1);   // partial buffer pb has been read out
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (elect_one()) {
                const uint32_t a_hi = smem_u32(smem + (size_t)s * stage_bytes);
                const uint32_t b_hi = a_hi + a_bytes;
                const uint32_t a_lo = smem_u32(lo_base + (size_t)sl * stage_bytes);
                const uint32_t b_lo = a_lo + a_bytes;
                const uint32_t d = tmem_base + (uint32_t)(pb * NT);
                // the two correction products first (tiny partial sums), then the main product
#pragma unroll
                for (int k = 0; k < TILE_K / UMMA_K; k++) {
                    const uint32_t koff = (uint32_t)k * UMMA_K * 4;   // 32 B per k-step inside the swizzle row
                    umma_tf32(d, umma_desc_k_sw128(a_lo + koff), umma_desc_k_sw128(b_hi + koff), idesc, (k > 0 || !first) ? 1u : 0u);
                    umma_tf32(d, umma_desc_k_sw128(a_hi + koff), umma_desc_k_sw128(b_lo + koff), idesc, 1u);
                }
#pragma unroll
                for (int k = 0; k < TILE_K / UMMA_K; k++) {
                    const uint32_t koff = (uint32_t)k * UMMA_K * 4;
                    umma_tf32(d, umma_desc_k_sw128(a_hi + koff), umma_desc_k_sw128(b_hi + koff), idesc, 1u);
                }
                umma_commit(raw_empty_bar(s));   // frees the stages when these MMAs have read them
                umma_commit(lo_empty_bar(sl));
                if (last) umma_commit(pfull_bar(pb));   // partial sums of this chunk of k-blocks complete
            }
            __syncwarp();
        }
    } else {
        // ------------------------------------------------ split workers / drain / epilogue
        const int t = threadIdx.x - 64;                      // 0..255
        const int q = warp & 3;                              // this warp may read TMEM lanes [32q, 32q+32)
        const int half = (warp - 2) >> 2;                    // ... and owns this half of the columns
        constexpr int NC = NT / 2;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * NC);
        float tot[NC];
#pragma unroll
        for (int j = 0; j < NC; j++) tot[j] = 0.f;
        auto drain = [&](int ch) {
            const int pb = ch & 1;
            mbar_wait(pfull_bar(pb), (ch >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            uint32_t r[NC];
#pragma unroll
            for (int c = 0; c < NC; c += 16) {   // all loads in flight, one wait
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                    : "=r"(r[c + 0]), "=r"(r[c + 1]), "=r"(r[c + 2]), "=r"(r[c + 3]), "=r"(r[c + 4]), "=r"(r[c + 5]),
                      "=r"(r[c + 6]), "=r"(r[c + 7]), "=r"(r[c + 8]), "=r"(r[c + 9]), "=r"(r[c + 10]), "=r"(r[c + 11]),
                      "=r"(r[c + 12]), "=r"(r[c + 13]), "=r"(r[c + 14]), "=r"(r[c + 15])
                    : "r"(taddr + (uint32_t)(pb * NT + c)));
            }
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int j = 0; j < NC; j++) tot[j] += __uint_as_float(r[j]);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(drained_bar(pb));
        };
        for (int kb = 0; kb < nkb; kb++) {
            const int s = kb % RAW_STAGES, sl = kb % LO_STAGES;
            mbar_wait(full_bar(s), (kb / RAW_STAGES) & 1);
            mbar_wait(lo_empty_bar(sl), ((kb / LO_STAGES) & 1) ^ 1);
            uint4* a_hi = reinterpret_cast<uint4*>(smem + (size_t)s * stage_bytes);
            uint4* b_hi = a_hi + a_bytes / 16;
            uint4* a_lo = reinterpret_cast<uint4*>(lo_base + (size_t)sl * stage_bytes);
            uint4* b_lo = a_lo + a_bytes / 16;
            auto split = [](uint4* hi, uint4* lo, int i) {
                uint4 v = hi[i], h, l;
                h.x = v.x & 0xffffe000u; h.y = v.y & 0xffffe000u; h.z = v.z & 0xffffe000u; h.w = v.w & 0xffffe000u;
                l.x = __float_as_uint(__uint_as_float(v.x) - __uint_as_float(h.x)) & 0xffffe000u;
                l.y = __float_as_uint(__uint_as_float(v.y) - __uint_as_float(h.y)) & 0xffffe000u;
                l.z = __float_as_uint(__uint_as_float(v.z) - __uint_as_float(h.z)) & 0xffffe000u;
                l.w = __float_as_uint(__uint_as_float(v.w) - __uint_as_float(h.w)) & 0xffffe000u;
                lo[i] = l;   // hi[i] keeps the raw value: the MMA ignores its low 13 mantissa bits (measured: bit-identical)
            };
#pragma unroll
            for (int i = 0; i < (TILE_M * TILE_K / 4) / SPLIT_THREADS; i++) split(a_hi, a_lo, t + i * SPLIT_THREADS);
#pragma unroll
            for (int i = 0; i < (NT * TILE_K / 4) / SPLIT_THREADS; i++) split(b_hi, b_lo, t + i * SPLIT_THREADS);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> visible to the MMA (async proxy)
            __syncwarp();
            if (lane == 0) mbar_arrive(ready_bar(sl));
            if (kb > 0 && kb % DRAIN_KB == 0) drain(kb / DRAIN_KB - 1);
        }
        drain((nkb - 1) / DRAIN_KB);
        // epilogue from registers: thread = half of one output row
        const int row = m0 + q * 32 + lane;
        const int c0 = half * NC;
        const int n_valid = min(NT, p.N - n0);
        if (p.tma_store) {
            // A thread owning a row would store with a 4*ldc-byte stride between lanes (one 32-byte
            // sector per lane and instruction: measured 12 us for a 128 x 192 tile).  Instead the tile is
            // staged in shared memory -- the operand rings are free now -- as NT/32 sub-tiles of
            // [128 rows x 128 bytes] in the 128-byte swizzle (conflict-free float4 writes) and written
            // by TMA, which also clips at the matrix edge.
            const int r = q * 32 + lane;
            const bool bias4 = p.bias && (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0;
#pragma unroll
            for (int c = 0; c < NC; c += 4) {
                float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
                if (bias4 && c0 + c + 4 <= n_valid) {
                    bv = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + c0 + c));
                } else if (p.bias) {
                    if (c0 + c + 0 < n_valid) bv.x = __ldg(p.bias + n0 + c0 + c + 0);
                    if (c0 + c + 1 < n_valid) bv.y = __ldg(p.bias + n0 + c0 + c + 1);
                    if (c0 + c + 2 < n_valid) bv.z = __ldg(p.bias + n0 + c0 + c + 2);
                    if (c0 + c + 3 < n_valid) bv.w = __ldg(p.bias + n0 + c0 + c + 3);
                }
                float4 o;
                o.x = apply_act(tot[c + 0] + bv.x, p.act);
                o.y = apply_act(tot[c + 1] + bv.y, p.act);
                o.z = apply_act(tot[c + 2] + bv.z, p.act);
                o.w = apply_act(tot[c + 3] + bv.w, p.act);
                const int col = c0 + c, sub = col >> 5, chunk = (col & 31) >> 2;
                *reinterpret_cast<float4*>(smem + (size_t)sub * (TILE_M * 128) + r * 128 + ((chunk ^ (r & 7)) << 4)) = o;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("bar.sync 1, %0;" ::"n"(SPLIT_THREADS) : "memory");
            if (threadIdx.x == 64) {
#pragma unroll
                for (int sub = 0; sub < NT / 32; sub++) {
                    if (n0 + sub * 32 < p.N)
                        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                                     ::"l"(&map_c), "r"(smem_u32(smem + (size_t)sub * (TILE_M * 128))), "r"(n0 + sub * 32), "r"(m0)
                                     : "memory");
                }
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // smem must outlive the reads
            }
        } else if (row < p.M) {
            float* crow = p.C + (int64_t)row * p.ldc + n0;
#pragma unroll
            for (int c = 0; c < NC; c++)
                if (c0 + c < n_valid)
                    crow[c0 + c] = apply_act(tot[c] + (p.bias ? __ldg(p.bias + n0 + c0 + c) : 0.f), p.act);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// rows x K fp32 matrix, row stride ld elements; box = 32 x box_rows, 128-byte swizzle, zero fill out of bounds
bool make_map(CUtensorMap* map, const float* base, int64_t rows, int64_t K, int64_t ld, int box_rows) {
    return make_map_2d(map, base, K, rows, ld, TILE_K, box_rows, true);
}

}  // namespace

extern "C" {

int mlb_linear_tc_supported(int32_t M, int32_t N, int32_t K, int64_t lda, int64_t ldw, int64_t ldc) {
    return M >= 1 && N >= 1 && K >= 1 && (lda % 4) == 0 && (ldw % 4) == 0 && lda >= K && ldw >= K && ldc >= N;
}

int mlb_linear_tc(const float* X, int64_t lda, const float* W, int64_t ldw, const float* bias, float* C, int64_t ldc,
                  int32_t M, int32_t N, int32_t K, int32_t act, void* stream) {
    if (!X || !W || !C) return MLB_EINVAL;
    if (!mlb_linear_tc_supported(M, N, K, lda, ldw, ldc)) return MLB_EINVAL;
    if ((reinterpret_cast<uintptr_t>(X) & 15) || (reinterpret_cast<uintptr_t>(W) & 15)) return MLB_EINVAL;
    // tile width: the per-k-block cost hardly depends on NT (the x tile dominates), so cover N with as few tiles as possible
    int NT = 32;
    for (int cand : {64, 128, 192})
        if ((N + cand - 1) / cand < (N + NT - 1) / NT) NT = cand;   // fewest tiles, then the narrowest
    const int raw = NT == 192 ? 3 : 4;
    const void* fn = NT == 32 ? (const void*)linear_tc_kernel<32, 4>
                   : NT == 64 ? (const void*)linear_tc_kernel<64, 4>
                   : NT == 128 ? (const void*)linear_tc_kernel<128, 4> : (const void*)linear_tc_kernel<192, 3>;
    const int n_tiles = (N + NT - 1) / NT;
    CUtensorMap mx, mw;
    if (!make_map(&mx, X, M, K, lda, TILE_M) || !make_map(&mw, W, N, K, ldw, NT)) return MLB_ECUDA;
    CUtensorMap mc = mx;   // placeholder when the TMA store cannot be used
    const int tma_store = (ldc % 4 == 0) && (reinterpret_cast<uintptr_t>(C) & 15) == 0 && make_map(&mc, C, M, N, ldc, TILE_M);
    TcParams p{C, bias, ldc, M, N, K, act, tma_store};
    const size_t smem = (size_t)(raw + LO_STAGES) * (TILE_M * TILE_K * 4 + (size_t)NT * TILE_K * 4) +
                        8 * (2 * raw + 2 * LO_STAGES + 6) + 1024;
    if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return MLB_ECUDA;
    dim3 grid(n_tiles, (M + TILE_M - 1) / TILE_M);
    void* args[] = {&mx, &mw, &mc, &p};
    if (cudaLaunchKernel(fn, grid, dim3(THREADS), args, smem, (cudaStream_t)stream) != cudaSuccess) return MLB_ECUDA;
    return cudaGetLastError() == cudaSuccess ? MLB_OK : MLB_ECUDA;
}

}  // extern "C"
