// Batched policy kernels behind include/marllb_b200_policy.h (QMIX / SAC-GRU, fp32).
//
// Reference modules: problem-05-qmix/src/{agent_network,mixing_network,qmix_agent}.py and
// problem-04-sac-gru/src/{networks,sac_agent}.py (paths under simulation-mode/).
#include <algorithm>
#include <mutex>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/marllb_b200.h"
#include "../../include/marllb_b200_policy.h"

namespace {

constexpr int BM = 64, BN = 64, BK = 16, TM = 4, TN = 4;  // 256 threads, 4x4 outputs each

// C = act(beta*C + A.B + bias), generic strides, fp32 FFMA, shared-memory tiled.
__global__ void __launch_bounds__(256)
gemm_kernel(const float* __restrict__ A, int64_t a_bs, int64_t a_rs, int64_t a_cs,
            const float* __restrict__ B, int64_t b_bs, int64_t b_rs, int64_t b_cs,
            float* __restrict__ C, int64_t c_bs, int64_t ldc, const float* __restrict__ bias,
            int64_t bias_bs, int M, int N, int K, float beta, int act, int splits, float* __restrict__ ws) {
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    // split-K (small outputs with a long reduction, e.g. M = 256 rows x K = 3000): z = batch * splits + split,
    // raw partial sums go to the workspace and splitk_reduce_kernel applies beta / bias / activation
    const int b = blockIdx.z / splits, sp = blockIdx.z - b * splits;
    const int kchunk = ((K + splits - 1) / splits + BK - 1) / BK * BK;
    const int k_lo = sp * kchunk, k_hi = min(K, k_lo + kchunk);
    A += (int64_t)b * a_bs;
    B += (int64_t)b * b_bs;
    C += (int64_t)b * c_bs;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int tid = threadIdx.x;
    const int tx = tid % (BN / TN), ty = tid / (BN / TN);  // 16 x 16
    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; i++)
#pragma unroll
        for (int j = 0; j < TN; j++) acc[i][j] = 0.f;
    const bool a_kfast = (a_cs == 1);  // k contiguous in A -> walk k fastest when loading
    const bool b_nfast = (b_cs == 1);  // n contiguous in B
    for (int k0 = k_lo; k0 < k_hi; k0 += BK) {
#pragma unroll
        for (int i = 0; i < (BM * BK) / 256; i++) {
            const int t = tid + i * 256;
            const int ml = a_kfast ? t / BK : t % BM;
            const int kl = a_kfast ? t % BK : t / BM;
            const int m = m0 + ml, k = k0 + kl;
            As[kl][ml] = (m < M && k < k_hi) ? A[(int64_t)m * a_rs + (int64_t)k * a_cs] : 0.f;
        }
#pragma unroll
        for (int i = 0; i < (BN * BK) / 256; i++) {
            const int t = tid + i * 256;
            const int nl = b_nfast ? t % BN : t / BK;
            const int kl = b_nfast ? t / BN : t % BK;
            const int n = n0 + nl, k = k0 + kl;
            Bs[kl][nl] = (n < N && k < k_hi) ? B[(int64_t)k * b_rs + (int64_t)n * b_cs] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; kk++) {
            float a[TM], bb[TN];
#pragma unroll
            for (int i = 0; i < TM; i++) a[i] = As[kk][ty * TM + i];
#pragma unroll
            for (int j = 0; j < TN; j++) bb[j] = Bs[kk][tx * TN + j];
#pragma unroll
            for (int i = 0; i < TM; i++)
#pragma unroll
                for (int j = 0; j < TN; j++) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
        }
        __syncthreads();
    }
    if (bias) bias += (int64_t)b * bias_bs;
#pragma unroll
    for (int i = 0; i < TM; i++) {
        const int m = m0 + ty * TM + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < TN; j++) {
            const int n = n0 + tx * TN + j;
            if (n >= N) continue;
            float v = acc[i][j];
            if (splits > 1) {
                ws[(((int64_t)sp * (gridDim.z / splits) + b) * M + m) * N + n] = v;
                continue;
            }
            if (bias) v += bias[n];
            if (beta != 0.f) v += beta * C[(int64_t)m * ldc + n];
            if (act == MLB_ACT_RELU) v = fmaxf(v, 0.f);
            else if (act == MLB_ACT_ABS) v = fabsf(v);
            C[(int64_t)m * ldc + n] = v;
        }
    }
}

// ---- skinny products of the MLP heads (fc3: 256 -> 1 and its two gradients), where a 64 x 64 tile is mostly padding
// C[m][n], n < N <= 8: one warp per output row, lanes stride the contraction, shuffle reduction
template <int NMAX>
__global__ void gemm_skinny_n_kernel(const float* __restrict__ A, int64_t a_rs, int64_t a_cs, const float* __restrict__ B,
                                     int64_t b_rs, int64_t b_cs, float* __restrict__ C, int64_t ldc,
                                     const float* __restrict__ bias, int M, int N, int K, float beta, int act) {
    const int m = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (m >= M) return;
    float acc[NMAX];
#pragma unroll
    for (int n = 0; n < NMAX; n++) acc[n] = 0.f;
    for (int k = lane; k < K; k += 32) {
        const float a = __ldg(A + (int64_t)m * a_rs + (int64_t)k * a_cs);
#pragma unroll
        for (int n = 0; n < NMAX; n++)
            if (n < N) acc[n] = fmaf(a, __ldg(B + (int64_t)k * b_rs + (int64_t)n * b_cs), acc[n]);
    }
#pragma unroll
    for (int n = 0; n < NMAX; n++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[n] += __shfl_xor_sync(0xffffffffu, acc[n], o);
    }
    if (lane < N) {
        float v = 0.f;
#pragma unroll
        for (int n = 0; n < NMAX; n++) v = lane == n ? acc[n] : v;
        if (bias) v += bias[lane];
        float* c = C + (int64_t)m * ldc + lane;
        if (beta != 0.f) v += beta * *c;
        if (act == MLB_ACT_RELU) v = fmaxf(v, 0.f);
        else if (act == MLB_ACT_ABS) v = fabsf(v);
        *c = v;
    }
}
// C[m][n], m < M <= 8: block = 32 columns x 32 contraction lanes (coalesced over n when b_cs == 1), shared-memory reduction
template <int MMAX>
__global__ void gemm_skinny_m_kernel(const float* __restrict__ A, int64_t a_rs, int64_t a_cs, const float* __restrict__ B,
                                     int64_t b_rs, int64_t b_cs, float* __restrict__ C, int64_t ldc,
                                     const float* __restrict__ bias, int M, int N, int K, float beta, int act) {
    __shared__ float part[32][MMAX][33];
    const int n = blockIdx.x * 32 + threadIdx.x;
    float acc[MMAX];
#pragma unroll
    for (int m = 0; m < MMAX; m++) acc[m] = 0.f;
    if (n < N) {
#pragma unroll 4
        for (int k = threadIdx.y; k < K; k += 32) {
            const float b = __ldg(B + (int64_t)k * b_rs + (int64_t)n * b_cs);
#pragma unroll
            for (int m = 0; m < MMAX; m++)
                if (m < M) acc[m] = fmaf(__ldg(A + (int64_t)m * a_rs + (int64_t)k * a_cs), b, acc[m]);
        }
    }
#pragma unroll
    for (int m = 0; m < MMAX; m++) part[threadIdx.y][m][threadIdx.x] = acc[m];
    __syncthreads();
    if (n < N && threadIdx.y < M) {
        const int m = threadIdx.y;
        float v = 0.f;
#pragma unroll
        for (int j = 0; j < 32; j++) v += part[j][m][threadIdx.x];
        if (bias) v += bias[n];
        float* c = C + (int64_t)m * ldc + n;
        if (beta != 0.f) v += beta * *c;
        if (act == MLB_ACT_RELU) v = fmaxf(v, 0.f);
        else if (act == MLB_ACT_ABS) v = fabsf(v);
        *c = v;
    }
}
// K <= 8 (outer products): one thread per output element
__global__ void gemm_thin_k_kernel(const float* __restrict__ A, int64_t a_rs, int64_t a_cs, const float* __restrict__ B,
                                   int64_t b_rs, int64_t b_cs, float* __restrict__ C, int64_t ldc,
                                   const float* __restrict__ bias, int M, int N, int K, float beta, int act) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= (int64_t)M * N) return;
    const int m = (int)(i / N), n = (int)(i - (int64_t)m * N);
    float v = 0.f;
    for (int k = 0; k < K; k++) v = fmaf(__ldg(A + (int64_t)m * a_rs + (int64_t)k * a_cs), __ldg(B + (int64_t)k * b_rs + (int64_t)n * b_cs), v);
    if (bias) v += bias[n];
    float* c = C + (int64_t)m * ldc + n;
    if (beta != 0.f) v += beta * *c;
    if (act == MLB_ACT_RELU) v = fmaxf(v, 0.f);
    else if (act == MLB_ACT_ABS) v = fabsf(v);
    *c = v;
}

// C = act(beta*C + sum_s ws[s] + bias), partial sums added in split order (deterministic)
__global__ void splitk_reduce_kernel(const float* __restrict__ ws, int splits, int batch, float* __restrict__ C,
                                     int64_t c_bs, int64_t ldc, const float* __restrict__ bias, int64_t bias_bs,
                                     int M, int N, float beta, int act) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t per = (int64_t)M * N;
    if (i >= per * batch) return;
    const int b = (int)(i / per);
    const int64_t r = i - (int64_t)b * per;
    const int m = (int)(r / N), n = (int)(r - (int64_t)m * N);
    float v = 0.f;
    for (int s = 0; s < splits; s++) v += ws[((int64_t)s * batch + b) * per + r];
    if (bias) v += bias[(int64_t)b * bias_bs + n];
    float* c = C + (int64_t)b * c_bs + (int64_t)m * ldc + n;
    if (beta != 0.f) v += beta * *c;
    if (act == MLB_ACT_RELU) v = fmaxf(v, 0.f);
    else if (act == MLB_ACT_ABS) v = fabsf(v);
    *c = v;
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

__global__ void gru_gates_fwd_kernel(const float* __restrict__ gi, const float* __restrict__ gh,
                                     const float* __restrict__ h, float* __restrict__ h_new,
                                     float* __restrict__ gates, int M, int H) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)M * H) return;
    const int m = (int)(i / H), c = (int)(i % H);
    const float* gim = gi + (int64_t)m * 3 * H;
    const float* ghm = gh + (int64_t)m * 3 * H;
    const float r = sigmoidf_(gim[c] + ghm[c]);
    const float z = sigmoidf_(gim[H + c] + ghm[H + c]);
    const float n = tanhf(gim[2 * H + c] + r * ghm[2 * H + c]);
    h_new[i] = (1.f - z) * n + z * h[i];
    if (gates) {
        float* gm = gates + (int64_t)m * 3 * H;
        gm[c] = r; gm[H + c] = z; gm[2 * H + c] = n;
    }
}

__global__ void gru_gates_bwd_kernel(const float* __restrict__ dh_new, const float* __restrict__ gates,
                                     const float* __restrict__ h, const float* __restrict__ gh,
                                     float* __restrict__ dgi, float* __restrict__ dgh,
                                     float* __restrict__ dh_direct, int M, int H) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)M * H) return;
    const int m = (int)(i / H), c = (int)(i % H);
    const float* gm = gates + (int64_t)m * 3 * H;
    const float r = gm[c], z = gm[H + c], n = gm[2 * H + c];
    const float g = dh_new[i];
    const float dn = g * (1.f - z);
    const float dz = g * (h[i] - n);
    const float dan = dn * (1.f - n * n);
    const float ghn = gh[(int64_t)m * 3 * H + 2 * H + c];
    const float dar = dan * ghn * r * (1.f - r);
    const float daz = dz * z * (1.f - z);
    float* dgim = dgi + (int64_t)m * 3 * H;
    float* dghm = dgh + (int64_t)m * 3 * H;
    dgim[c] = dar; dgim[H + c] = daz; dgim[2 * H + c] = dan;
    dghm[c] = dar; dghm[H + c] = daz; dghm[2 * H + c] = dan * r;
    dh_direct[i] = g * z;
}

// ---- the GRU time loop of an update in ONE launch (forward) and one more (backward through time).
// QMIXAgent.update unrolls T = 50 steps per agent (qmix_agent.py:217-224, 246-253): launched step by step that is ~10
// kernels per step and agent, each microseconds of work.  Batch rows are independent, so a block takes RB rows through
// all T steps with the recurrent weights resident in shared memory (3H x H floats: 48 KB at H = 64) and the hidden
// state never leaving the SM.  Same arithmetic as the per-step kernels (gemm accumulation order k = 0..H-1 with fmaf,
// bias added last; gru_gates_fwd/bwd formulas), so the two forms agree to fp32 rounding.
constexpr int GRU_SEQ_RB = 4;   // batch rows per block

// hs[t] = GRU(gi_all[t], hs[t-1]);  saves what backward needs (nullable): hprev[t], ghs[t] = h W_hh^T + b_hh, gates[t]
__global__ void gru_seq_fwd_kernel(const float* __restrict__ gi_all, const float* __restrict__ W_hh,
                                   const float* __restrict__ b_hh, const float* __restrict__ h0, float* __restrict__ hs,
                                   float* __restrict__ hprev, float* __restrict__ ghs, float* __restrict__ gates, int T, int B,
                                   int H) {
    extern __shared__ __align__(16) float gsm[];
    const int H3 = 3 * H;
    const int H3P = H3 + 1;                // padded row: the transposing stores below (k consecutive) hit distinct banks
    float* WT = gsm;                       // [H][3H+1]: WT[k][j] = W_hh[j][k] (threads j consecutive: conflict-free)
    float* h_s = WT + (size_t)H * H3P;     // [RB][H]
    float* gh_s = h_s + GRU_SEQ_RB * H;    // [RB][3H]
    const int tid = threadIdx.x, nt = blockDim.x;     // nt = 3H
    const int b0 = blockIdx.x * GRU_SEQ_RB;
    const int nr = min(GRU_SEQ_RB, B - b0);
    if ((H & 3) == 0) {                    // 128-bit loads, several in flight (T = 1 calls are all prologue)
        const float4* W4 = reinterpret_cast<const float4*>(W_hh);
#pragma unroll 4
        for (int i = tid; i < H3 * H / 4; i += nt) {
            const float4 w = __ldg(W4 + i);
            const int j = (i * 4) / H, k = i * 4 - j * H;
            float* dst = WT + (size_t)k * H3P + j;
            dst[0] = w.x; dst[H3P] = w.y; dst[2 * H3P] = w.z; dst[3 * H3P] = w.w;
        }
    } else {
        for (int i = tid; i < H3 * H; i += nt) {
            const int j = i / H, k = i - j * H;
            WT[(size_t)k * H3P + j] = __ldg(W_hh + i);
        }
    }
    for (int i = tid; i < GRU_SEQ_RB * H; i += nt) {
        const int r = i / H, c = i - r * H;
        h_s[i] = r < nr ? __ldg(h0 + (size_t)(b0 + r) * H + c) : 0.f;
    }
    const float bj = __ldg(b_hh + tid);
    __syncthreads();
    for (int t = 0; t < T; t++) {
        // gh[r][j] = sum_k h[r][k] W_hh[j][k] + b_hh[j], thread = j
        float acc[GRU_SEQ_RB];
#pragma unroll
        for (int r = 0; r < GRU_SEQ_RB; r++) acc[r] = 0.f;
        for (int k = 0; k < H; k++) {
            const float w = WT[(size_t)k * H3P + tid];
#pragma unroll
            for (int r = 0; r < GRU_SEQ_RB; r++) acc[r] = fmaf(h_s[r * H + k], w, acc[r]);
        }
#pragma unroll
        for (int r = 0; r < GRU_SEQ_RB; r++) {
            const float v = acc[r] + bj;
            gh_s[r * H3 + tid] = v;
            if (ghs && r < nr) ghs[((size_t)t * B + b0 + r) * H3 + tid] = v;
        }
        __syncthreads();
        // gates (gate order r, z, n) and the new hidden state, thread = (row, column)
        for (int i = tid; i < nr * H; i += nt) {
            const int r = i / H, c = i - r * H;
            const size_t row = (size_t)t * B + b0 + r;
            const float* gim = gi_all + row * H3;
            const float* ghm = gh_s + r * H3;
            const float rg = sigmoidf_(__ldg(gim + c) + ghm[c]);
            const float z = sigmoidf_(__ldg(gim + H + c) + ghm[H + c]);
            const float n = tanhf(__ldg(gim + 2 * H + c) + rg * ghm[2 * H + c]);
            const float hold = h_s[i];
            const float hn = (1.f - z) * n + z * hold;
            if (hprev) hprev[row * H + c] = hold;
            hs[row * H + c] = hn;
            if (gates) {
                float* gm = gates + row * H3;
                gm[c] = rg; gm[H + c] = z; gm[2 * H + c] = n;
            }
            h_s[i] = hn;
        }
        __syncthreads();
    }
}

// backward through time: dgi_all[t], dgh_all[t] for every step and the gradient w.r.t. h0
__global__ void gru_seq_bwd_kernel(const float* __restrict__ dhs, const float* __restrict__ gates,
                                   const float* __restrict__ hprev, const float* __restrict__ ghs,
                                   const float* __restrict__ W_hh, float* __restrict__ dgi_all, float* __restrict__ dgh_all,
                                   float* __restrict__ dh0, int T, int B, int H) {
    extern __shared__ __align__(16) float gsm[];
    const int H3 = 3 * H;
    float* W = gsm;                            // [3H][H] as stored (threads k consecutive: conflict-free)
    float* dh_s = W + (size_t)H3 * H;          // [RB][H] gradient flowing into step t from step t+1
    float* dgh_s = dh_s + GRU_SEQ_RB * H;      // [RB][3H]
    float* part = dgh_s + GRU_SEQ_RB * H3;     // [3][RB][H] partial products per gate block
    const int tid = threadIdx.x, nt = blockDim.x;     // nt = 3H
    const int b0 = blockIdx.x * GRU_SEQ_RB;
    const int nr = min(GRU_SEQ_RB, B - b0);
    if ((H & 3) == 0) {
#pragma unroll 4
        for (int i = tid; i < H3 * H / 4; i += nt) reinterpret_cast<float4*>(W)[i] = __ldg(reinterpret_cast<const float4*>(W_hh) + i);
    } else {
        for (int i = tid; i < H3 * H; i += nt) W[i] = __ldg(W_hh + i);
    }
    for (int i = tid; i < GRU_SEQ_RB * H; i += nt) dh_s[i] = 0.f;
    for (int i = tid; i < GRU_SEQ_RB * H3; i += nt) dgh_s[i] = 0.f;
    __syncthreads();
    const int g = tid / H, k = tid - g * H;    // gate block and hidden column of this thread in the product below
    for (int t = T - 1; t >= 0; t--) {
        for (int i = tid; i < nr * H; i += nt) {
            const int r = i / H, c = i - r * H;
            const size_t row = (size_t)t * B + b0 + r;
            const float* gm = gates + row * H3;
            const float rg = __ldg(gm + c), z = __ldg(gm + H + c), n = __ldg(gm + 2 * H + c);
            const float gr = __ldg(dhs + row * H + c) + dh_s[i];
            const float dn = gr * (1.f - z);
            const float dz = gr * (__ldg(hprev + row * H + c) - n);
            const float dan = dn * (1.f - n * n);
            const float ghn = __ldg(ghs + row * H3 + 2 * H + c);
            const float dar = dan * ghn * rg * (1.f - rg);
            const float daz = dz * z * (1.f - z);
            float* dgim = dgi_all + row * H3;
            float* dghm = dgh_all + row * H3;
            dgim[c] = dar; dgim[H + c] = daz; dgim[2 * H + c] = dan;
            const float dghn = dan * rg;
            dghm[c] = dar; dghm[H + c] = daz; dghm[2 * H + c] = dghn;
            dgh_s[r * H3 + c] = dar; dgh_s[r * H3 + H + c] = daz; dgh_s[r * H3 + 2 * H + c] = dghn;
            dh_s[i] = gr * z;                  // direct path h_{t-1} -> h_t
        }
        __syncthreads();
        // dh_prev[r][k] = dh_direct + sum_j dgh[r][j] W_hh[j][k]: thread (g, k) sums gate block g
        float acc[GRU_SEQ_RB];
#pragma unroll
        for (int r = 0; r < GRU_SEQ_RB; r++) acc[r] = 0.f;
        for (int jj = 0; jj < H; jj++) {
            const float w = W[(size_t)(g * H + jj) * H + k];
#pragma unroll
            for (int r = 0; r < GRU_SEQ_RB; r++) acc[r] = fmaf(dgh_s[r * H3 + g * H + jj], w, acc[r]);
        }
#pragma unroll
        for (int r = 0; r < GRU_SEQ_RB; r++) part[(g * GRU_SEQ_RB + r) * H + k] = acc[r];
        __syncthreads();
        for (int i = tid; i < GRU_SEQ_RB * H; i += nt)
            dh_s[i] += (part[i] + part[GRU_SEQ_RB * H + i]) + part[2 * GRU_SEQ_RB * H + i];
        __syncthreads();
    }
    if (dh0)
        for (int i = tid; i < nr * H; i += nt) dh0[(size_t)(b0 + i / H) * H + (i % H)] = dh_s[i];
}

__global__ void relu_bwd_kernel(const float* __restrict__ y, const float* __restrict__ dy, float* __restrict__ dx, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dx[i] = y[i] > 0.f ? dy[i] : 0.f;
}

__global__ void abs_bwd_kernel(const float* __restrict__ pre, const float* __restrict__ dy, float* __restrict__ dx, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const float p = pre[i];
        dx[i] = p > 0.f ? dy[i] : (p < 0.f ? -dy[i] : 0.f);  // torch.abs: grad * sign(x)
    }
}

// db[n] = beta*db[n] + sum_m dy[m][n]; one block per 32 columns, 32 row-lanes
__global__ void colsum_kernel(const float* __restrict__ dy, float* __restrict__ db, int M, int N, int64_t ld, float beta) {
    __shared__ float part[32][33];
    const int n = blockIdx.x * 32 + threadIdx.x;
    float s = 0.f;
    if (n < N) {
#pragma unroll 4
        for (int m = threadIdx.y; m < M; m += 32) s += __ldg(dy + (int64_t)m * ld + n);
    }
    part[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && n < N) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < 32; k++) t += part[k][threadIdx.x];
        db[n] = (beta != 0.f ? beta * db[n] : 0.f) + t;
    }
}

__global__ void axpby_kernel(float a, const float* __restrict__ x, float b, float* __restrict__ y, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = a * x[i] + b * y[i];
}

__global__ void sumsq_kernel(const float* __restrict__ x, int64_t n, double* out) {
    double s = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double v = (double)x[i];
        s += v * v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, s);
}

__global__ void scale_kernel(float* __restrict__ x, int64_t n, const double* __restrict__ norm_sq, float max_norm) {
    // torch.nn.utils.clip_grad_norm_: coef = max_norm / (total_norm + 1e-6), clamped to 1
    const float total = (float)sqrt(*norm_sq);
    float coef = max_norm / (total + 1e-6f);
    coef = coef > 1.f ? 1.f : coef;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] *= coef;
}

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, int64_t n, float beta1, float beta2, float eps,
                            float step_size, float bc2_sqrt) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float gi = g[i];
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;        // exp_avg.lerp_(grad, 1-beta1)
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;   // exp_avg_sq.mul_(beta2).addcmul_(g,g,1-beta2)
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= step_size * (mi / denom);
}

// Adam with the step counter on the device, so that an optimiser step can be replayed from a CUDA graph:
// the prologue advances the counter and derives the two bias-correction coefficients from it.
__global__ void adam_prep_kernel(int32_t* __restrict__ step, float lr, float beta1, float beta2, float* __restrict__ coef) {
    const int t = step[0] + 1;
    step[0] = t;
    const double bc1 = 1.0 - pow((double)beta1, (double)t);
    const double bc2 = 1.0 - pow((double)beta2, (double)t);
    coef[0] = (float)((double)lr / bc1);
    coef[1] = (float)sqrt(bc2);
}
__global__ void adam_dev_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                float* __restrict__ v, int64_t n, float beta1, float beta2, float eps,
                                const float* __restrict__ coef) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float step_size = coef[0], bc2_sqrt = coef[1];
    const float gi = g[i];
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= step_size * (mi / denom);
}

__global__ void egreedy_kernel(const float* __restrict__ q, const float* __restrict__ u, const int32_t* __restrict__ rnd,
                               float epsilon, int32_t* __restrict__ action, float* __restrict__ q_sel, int M, int K) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    const float* qm = q + (int64_t)m * K;
    int best = 0;
    float bv = qm[0];
    for (int k = 1; k < K; k++)
        if (qm[k] > bv) { bv = qm[k]; best = k; }   // first maximum
    int a = best;
    if (u && u[m] < epsilon) a = rnd[m];            // qmix_agent.py:159-161
    action[m] = a;
    if (q_sel) q_sel[m] = qm[a];
}

// QMIX action (one server index per agent, rl_controller.py:314-321: weight on the chosen server) ->
// the env's per-server discrete action: `hot` at the chosen server of each agent, `cold` elsewhere
__global__ void onehot_action_kernel(const int32_t* __restrict__ action, int M, int Sa, int stride, uint8_t hot, uint8_t cold,
                                     uint8_t* __restrict__ out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= (int64_t)M * Sa) return;
    const int m = (int)(i / Sa), j = (int)(i - (int64_t)m * Sa);
    out[i] = action[(int64_t)m * stride] == j ? hot : cold;
}

__global__ void row_max_kernel(const float* __restrict__ q, float* __restrict__ out, int32_t* __restrict__ arg, int M, int K) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    const float* qm = q + (int64_t)m * K;
    int best = 0;
    float bv = qm[0];
    for (int k = 1; k < K; k++)
        if (qm[k] > bv) { bv = qm[k]; best = k; }
    out[m] = bv;
    if (arg) arg[m] = best;
}

// one warp per sample
__global__ void mixer_fwd_kernel(const float* __restrict__ q, const float* __restrict__ w1, const float* __restrict__ b1,
                                 const float* __restrict__ w2, const float* __restrict__ b2, float* __restrict__ q_tot,
                                 float* __restrict__ hidden_out, int M, int A, int E) {
    const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (m >= M) return;
    float acc = 0.f;
    for (int e = lane; e < E; e += 32) {
        float pre = b1[(int64_t)m * E + e];
        for (int a = 0; a < A; a++) pre = fmaf(q[(int64_t)m * A + a], w1[((int64_t)m * A + a) * E + e], pre);
        const float hdn = pre > 0.f ? pre : expm1f(pre);   // F.elu, alpha = 1
        if (hidden_out) hidden_out[(int64_t)m * E + e] = hdn;
        acc = fmaf(hdn, w2[(int64_t)m * E + e], acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) q_tot[m] = acc + b2[m];
}

__global__ void mixer_bwd_kernel(const float* __restrict__ dq_tot, const float* __restrict__ q, const float* __restrict__ w1,
                                 const float* __restrict__ w2, const float* __restrict__ hidden, float* __restrict__ dq,
                                 float* __restrict__ dw1, float* __restrict__ db1, float* __restrict__ dw2,
                                 float* __restrict__ db2, int M, int A, int E) {
    const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (m >= M) return;
    const float g = dq_tot[m];
    if (lane == 0) db2[m] = g;
    for (int a = 0; a < A; a++) {
        float s = 0.f;
        for (int e = lane; e < E; e += 32) {
            const float hdn = hidden[(int64_t)m * E + e];
            const float dpre = g * w2[(int64_t)m * E + e] * (hdn > 0.f ? 1.f : hdn + 1.f);
            if (a == 0) {
                dw2[(int64_t)m * E + e] = g * hdn;
                db1[(int64_t)m * E + e] = dpre;
            }
            dw1[((int64_t)m * A + a) * E + e] = q[(int64_t)m * A + a] * dpre;
            s = fmaf(w1[((int64_t)m * A + a) * E + e], dpre, s);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) dq[(int64_t)m * A + a] = s;
    }
}

// one warp per sample
__global__ void tanh_gauss_fwd_kernel(const float* __restrict__ mean, const float* __restrict__ lsr, const float* __restrict__ eps,
                                      float lo, float hi, float scale, float bias, float* __restrict__ action,
                                      float* __restrict__ logp, float* __restrict__ mean_action, int M, int A) {
    const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (m >= M) return;
    float lp = 0.f;
    for (int a = lane; a < A; a += 32) {
        const int64_t i = (int64_t)m * A + a;
        const float mu = mean[i];
        const float ls = fminf(fmaxf(lsr[i], lo), hi);         // networks.py:108
        const float e = eps ? eps[i] : 0.f;
        const float x = mu + expf(ls) * e;                     // rsample
        const float y = tanhf(x);
        if (action) action[i] = y * scale + bias;
        if (mean_action) mean_action[i] = tanhf(mu) * scale + bias;
        // Normal.log_prob(x) - log(scale*(1-y^2)+1e-6)          networks.py:138-141
        lp += -0.5f * e * e - ls - 0.91893853320467274178f - logf(scale * (1.f - y * y) + 1e-6f);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lp += __shfl_xor_sync(0xffffffffu, lp, o);
    if (lane == 0 && logp) logp[m] = lp;
}

__global__ void tanh_gauss_bwd_kernel(const float* __restrict__ mean, const float* __restrict__ lsr, const float* __restrict__ eps,
                                      float lo, float hi, float scale, const float* __restrict__ d_action,
                                      const float* __restrict__ d_logp, float* __restrict__ d_mean,
                                      float* __restrict__ d_lsr, int M, int A) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)M * A) return;
    const int m = (int)(i / A);
    const float raw = lsr[i];
    const float ls = fminf(fmaxf(raw, lo), hi);
    const float sd = expf(ls), e = eps[i];
    const float y = tanhf(mean[i] + sd * e);
    const float omy2 = 1.f - y * y;
    const float gl = d_logp ? d_logp[m] : 0.f;
    const float ga = d_action ? d_action[i] : 0.f;
    // d/dx of -log(scale*(1-y^2)+1e-6) = 2*scale*y*(1-y^2) / (scale*(1-y^2)+1e-6)
    const float dx = ga * scale * omy2 + gl * (2.f * scale * y * omy2) / (scale * omy2 + 1e-6f);
    d_mean[i] = dx;
    const float dls = dx * sd * e - gl;
    d_lsr[i] = (raw >= lo && raw <= hi) ? dls : 0.f;          // torch.clamp passes gradient inside [lo, hi]
}

__global__ void abs_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = fabsf(x[i]);
}

__device__ __forceinline__ double block_sum(double v, double* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x < 32) {
        t = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    }
    __syncthreads();
    return t;  // valid in thread 0
}

// single block: B*T is small (<= a few thousand)
__global__ void qmix_td_loss_kernel(const float* __restrict__ q_tot, const float* __restrict__ tq, const float* __restrict__ rsum,
                                    const float* __restrict__ done, const int32_t* __restrict__ seq_len, float gamma,
                                    float* __restrict__ targets, float* __restrict__ dq, double* __restrict__ stats, int B, int T) {
    __shared__ double sh[32];
    __shared__ double s_msum;
    const int n = B * T;
    double msum = 0.0, lsum = 0.0, qsum = 0.0, tsum = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int b = i / T, t = i % T;
        const float shifted = t + 1 < T ? tq[i + 1] : 0.f;                   // qmix_agent.py:264-265
        const float y = rsum[i] + gamma * (1.f - done[i]) * shifted;         // :267-268
        targets[i] = y;
        const float mask = t < seq_len[b] ? 1.f : 0.f;                       // :271-273
        const float df = q_tot[i] - y;
        msum += mask;
        lsum += (double)(df * df * mask);
        qsum += q_tot[i];
        tsum += y;
    }
    const double M = block_sum(msum, sh);
    if (threadIdx.x == 0) s_msum = M;
    const double L = block_sum(lsum, sh);
    const double Qs = block_sum(qsum, sh);
    const double Ts = block_sum(tsum, sh);
    __syncthreads();
    const float inv = (float)(1.0 / s_msum);
    if (threadIdx.x == 0) {
        stats[0] = L / s_msum;
        stats[1] = Qs / n;
        stats[2] = Ts / n;
    }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int b = i / T, t = i % T;
        const float mask = t < seq_len[b] ? 1.f : 0.f;
        dq[i] = 2.f * (q_tot[i] - targets[i]) * mask * inv;
    }
}

__global__ void sac_q_target_kernel(const float* __restrict__ r, const float* __restrict__ d, const float* __restrict__ q1n,
                                    const float* __restrict__ q2n, const float* __restrict__ lp, const float* __restrict__ alpha,
                                    float gamma, float* __restrict__ y, int M) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < M) y[i] = r[i] + (1.f - d[i]) * gamma * (fminf(q1n[i], q2n[i]) - alpha[0] * lp[i]);
}

__global__ void mse_loss_kernel(const float* __restrict__ q, const float* __restrict__ y, float* __restrict__ dq,
                                double* __restrict__ loss, int M) {
    __shared__ double sh[32];
    double s = 0.0;
    for (int i = threadIdx.x; i < M; i += blockDim.x) {
        const float df = q[i] - y[i];
        s += (double)(df * df);
        dq[i] = 2.f * df / (float)M;
    }
    const double t = block_sum(s, sh);
    if (threadIdx.x == 0) *loss = t / M;
}

__global__ void sac_policy_loss_kernel(const float* __restrict__ lp, const float* __restrict__ q1, const float* __restrict__ q2,
                                       const float* __restrict__ alpha, float* __restrict__ dlp, float* __restrict__ dq1,
                                       float* __restrict__ dq2, double* __restrict__ loss, int M) {
    __shared__ double sh[32];
    double s = 0.0;
    const float a = alpha[0], inv = 1.f / (float)M;
    for (int i = threadIdx.x; i < M; i += blockDim.x) {
        const bool first = q1[i] <= q2[i];
        s += (double)(a * lp[i] - (first ? q1[i] : q2[i]));
        dlp[i] = a * inv;
        dq1[i] = first ? -inv : 0.f;
        dq2[i] = first ? 0.f : -inv;
    }
    const double t = block_sum(s, sh);
    if (threadIdx.x == 0) *loss = t / M;
}

__global__ void sac_alpha_loss_kernel(const float* __restrict__ lp, const float* __restrict__ log_alpha, float target_entropy,
                                      float* __restrict__ dla, double* __restrict__ loss, int M) {
    __shared__ double sh[32];
    double s = 0.0;
    for (int i = threadIdx.x; i < M; i += blockDim.x) s += (double)(lp[i] + target_entropy);
    const double t = block_sum(s, sh);
    if (threadIdx.x == 0) {
        dla[0] = (float)(-t / M);
        *loss = -(double)log_alpha[0] * t / M;
    }
}

__global__ void exp_scalar_kernel(const float* x, float* y) { y[0] = expf(x[0]); }

inline int ok() { return cudaGetLastError() == cudaSuccess ? MLB_OK : MLB_ECUDA; }
inline unsigned nblk(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

}  // namespace

// ---------------------------------------------------------------------------------------------
// Original-paper agents (src/lb/sac_qmix.py, src/lb/sac_gru_discrete.py): multi-head categorical
// outputs.  One thread per row of n <= 64 classes (n = discretised weight levels per head).
__global__ void softmax_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int64_t rows, int n) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const float* xr = x + r * n;
    float mx = xr[0];
    for (int k = 1; k < n; k++) mx = fmaxf(mx, xr[k]);
    float s = 0.f;
    for (int k = 0; k < n; k++) s += expf(xr[k] - mx);
    const float inv = 1.f / s;
    for (int k = 0; k < n; k++) y[r * n + k] = expf(xr[k] - mx) * inv;
}

// dx = y * (dy - sum_k dy_k y_k)
__global__ void softmax_bwd_kernel(const float* __restrict__ y, const float* __restrict__ dy, float* __restrict__ dx,
                                   int64_t rows, int n) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    float dot = 0.f;
    for (int k = 0; k < n; k++) dot = fmaf(dy[r * n + k], y[r * n + k], dot);
    for (int k = 0; k < n; k++) dx[r * n + k] = y[r * n + k] * (dy[r * n + k] - dot);
}

// out[row] = [ x[row][0:F] | one_hot(action[row][h], n) for h < heads ]   (sac_qmix.py:231-236)
__global__ void concat_onehot_kernel(const float* __restrict__ x, const int32_t* __restrict__ action, float* __restrict__ out,
                                     int64_t rows, int F, int heads, int n) {
    const int W = F + heads * n;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * W) return;
    const int64_t r = i / W;
    const int c = (int)(i - r * W);
    float v;
    if (c < F) {
        v = x[r * F + c];
    } else {
        const int h = (c - F) / n, k = (c - F) - h * n;
        v = action[r * heads + h] == k ? 1.f : 0.f;
    }
    out[i] = v;
}

// Categorical over rows of probabilities: inverse-CDF draw from a caller-supplied uniform (u nullable: argmax,
// first maximum like np.argmax), log-probability of the drawn class, gather of a given class.
__global__ void categorical_kernel(const float* __restrict__ p, const float* __restrict__ u, const int32_t* __restrict__ given,
                                   int32_t* __restrict__ action, float* __restrict__ logp, float* __restrict__ psel,
                                   int64_t rows, int n) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const float* pr = p + r * n;
    int a;
    if (given) {
        a = given[r];
    } else if (u) {
        float tot = 0.f;
        for (int k = 0; k < n; k++) tot += pr[k];
        const float cut = u[r] * tot;
        float c = 0.f;
        a = n - 1;
        for (int k = 0; k < n; k++) {
            c += pr[k];
            if (cut < c) { a = k; break; }
        }
    } else {
        a = 0;
        for (int k = 1; k < n; k++) if (pr[k] > pr[a]) a = k;
    }
    if (action) action[r] = a;
    if (logp) logp[r] = logf(pr[a]);                       // Categorical.log_prob
    if (psel) psel[r] = pr[a];                             // torch.gather(agent_outs, -1, action)
}

// gradient of sum_r g[r/group] * log p[r][a_r] w.r.t. the LOGITS of the softmax that produced p:
// dlogits[r][k] = g * ((k == a_r) - p[r][k]); `group` consecutive rows (the heads of one sample) share one g
__global__ void logprob_bwd_kernel(const float* __restrict__ p, const int32_t* __restrict__ action, const float* __restrict__ g,
                                   float* __restrict__ dlogits, int64_t rows, int n, int group) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * n) return;
    const int64_t r = i / n;
    const int k = (int)(i - r * n);
    dlogits[i] = g[r / group] * ((action[r] == k ? 1.f : 0.f) - p[i]);
}

// scatter of per-row gradients into the class that was chosen: d[r][k] = (k == a_r) ? g[r] : 0
__global__ void scatter_class_kernel(const float* __restrict__ g, const int32_t* __restrict__ action, float* __restrict__ d,
                                     int64_t rows, int n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * n) return;
    const int64_t r = i / n;
    d[i] = action[r] == (int)(i - r * n) ? g[r] : 0.f;
}

// WeightedQMixingNetwork.forward (mixing_network.py:231-246): q_tot[m] = sum_a q[m][a] * w[m][a]; one thread per row
__global__ void weighted_sum_fwd_kernel(const float* __restrict__ q, const float* __restrict__ w, float* __restrict__ out,
                                        int M, int A) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    float s = 0.f;
    for (int a = 0; a < A; a++) s += q[(int64_t)m * A + a] * w[(int64_t)m * A + a];
    out[m] = s;
}
__global__ void weighted_sum_bwd_kernel(const float* __restrict__ g, const float* __restrict__ q, const float* __restrict__ w,
                                        float* __restrict__ dq, float* __restrict__ dw, int64_t n, int A) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float gm = g[i / A];
    dq[i] = gm * w[i];
    dw[i] = gm * q[i];
}

// sac_qmix.py:449-460 _build_td_lambda_targets: backward recursion over the sequence, one thread per batch row
__global__ void td_lambda_kernel(const float* __restrict__ reward, const float* __restrict__ tq, float* __restrict__ ret,
                                 float gamma, float lam, int B, int T) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float* r = reward + (int64_t)b * T;
    const float* q = tq + (int64_t)b * T;
    float* o = ret + (int64_t)b * T;
    float nxt = q[T - 1];
    o[T - 1] = nxt;
    for (int t = T - 2; t >= 0; t--) {
        // torch evaluates td_lambda * gamma (Python floats, double) first, then float32 tensor ops
        const float v = __fadd_rn(__fmul_rn((float)((double)lam * (double)gamma), nxt),
                                  __fadd_rn(r[t], __fmul_rn((float)((1.0 - (double)lam) * (double)gamma), q[t + 1])));
        o[t] = v;
        nxt = v;
    }
}

// sac_gru_discrete.py:299-300: r <- scale * (r - mean_b r) / (std_b r + 1e-6) per sequence position
// (unbiased std over the batch dimension); one thread per position t
__global__ void reward_norm_kernel(const float* __restrict__ r, float* __restrict__ out, float scale, int B, int T) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    double s = 0.0;
    for (int b = 0; b < B; b++) s += (double)r[(int64_t)b * T + t];
    const double mean = s / B;
    double ss = 0.0;
    for (int b = 0; b < B; b++) {
        const double d = (double)r[(int64_t)b * T + t] - mean;
        ss += d * d;
    }
    const float sd = (float)sqrt(ss / (B - 1));
    const float mf = (float)mean;
    for (int b = 0; b < B; b++) out[(int64_t)b * T + t] = scale * (r[(int64_t)b * T + t] - mf) / (sd + 1e-6f);
}

// sac_gru_discrete.py:316-319: y = r + gamma * (min(q1, q2) - alpha * logp_next)   (no done flag in that trainer)
__global__ void dsac_q_target_kernel(const float* __restrict__ r, const float* __restrict__ q1n, const float* __restrict__ q2n,
                                     const float* __restrict__ lp, const float* __restrict__ alpha, float gamma,
                                     float* __restrict__ y, int M) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < M) y[i] = r[i] + gamma * (fminf(q1n[i], q2n[i]) - alpha[0] * lp[i]);
}

// ---- device-resident replay ring (rollout.DeviceReplay; reference: ReplayBuffer.push / sample,
// problem-04-sac-gru/src/replay_buffer.py:35-94, one transition per Python call into a host deque).
struct ReplayPtrs {
    float* state; float* action; float* next_state; float* hidden; float* reward; float* done;
};
__device__ __forceinline__ void replay_copy_row(float* dst, const float* src, int n) {
    if ((n & 3) == 0) {
        for (int i = threadIdx.x; i < n / 4; i += blockDim.x)
            reinterpret_cast<float4*>(dst)[i] = __ldg(reinterpret_cast<const float4*>(src) + i);
    } else {
        for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = __ldg(src + i);
    }
}
// E transitions -> ring rows (pos + e) % capacity; one block per transition
__global__ void replay_push_kernel(const float* __restrict__ state, const float* __restrict__ action,
                                   const double* __restrict__ reward, const float* __restrict__ next_state,
                                   const uint8_t* __restrict__ done, const float* __restrict__ hidden, ReplayPtrs r,
                                   const int64_t* __restrict__ pos, int capacity, int sd, int ad, int hd) {
    const int e = blockIdx.x;
    const int64_t row = (*pos + e) % capacity;
    replay_copy_row(r.state + row * sd, state + (int64_t)e * sd, sd);
    replay_copy_row(r.next_state + row * sd, next_state + (int64_t)e * sd, sd);
    replay_copy_row(r.action + row * ad, action + (int64_t)e * ad, ad);
    replay_copy_row(r.hidden + row * hd, hidden + (int64_t)e * hd, hd);
    if (threadIdx.x == 0) {
        r.reward[row] = (float)reward[e];
        r.done[row] = done[e] ? 1.f : 0.f;
    }
}
__global__ void replay_advance_kernel(int64_t* pos, int n, int capacity) { *pos = (*pos + n) % capacity; }
// batch rows idx[b] of the ring -> contiguous batch tensors
__global__ void replay_gather_kernel(ReplayPtrs r, const int64_t* __restrict__ idx, float* __restrict__ state,
                                     float* __restrict__ action, float* __restrict__ reward, float* __restrict__ next_state,
                                     float* __restrict__ done, float* __restrict__ hidden, int sd, int ad, int hd) {
    const int b = blockIdx.x;
    const int64_t row = idx[b];
    replay_copy_row(state + (int64_t)b * sd, r.state + row * sd, sd);
    replay_copy_row(next_state + (int64_t)b * sd, r.next_state + row * sd, sd);
    replay_copy_row(action + (int64_t)b * ad, r.action + row * ad, ad);
    replay_copy_row(hidden + (int64_t)b * hd, r.hidden + row * hd, hd);
    if (threadIdx.x == 0) {
        reward[b] = r.reward[row];
        done[b] = r.done[row];
    }
}

// Workspace slot of the calling host thread (split-K partial tiles): see mlb_set_workspace_slot in the header.
static thread_local int g_ws_slot = 0;
extern "C" int mlb_set_workspace_slot(int32_t slot) {
    if (slot < 0 || slot >= MLB_WS_SLOTS) return MLB_EINVAL;
    g_ws_slot = slot;
    return MLB_OK;
}
extern "C" int mlb_get_workspace_slot(void) { return g_ws_slot; }

// Split-K workspaces: [kind: 0 = FFMA gemm_kernel, 1 = gemm_tc_kernel][device][slot], grown outside stream capture only
// (cudaMalloc is not capturable); an outgrown buffer is left alone, queued work may still use it.
static float* g_ws_ptr[2][64][MLB_WS_SLOTS];
static size_t g_ws_cap[2][64][MLB_WS_SLOTS];
static std::mutex g_ws_mu;
static float* ws_grow(int kind, int dev, int slot, size_t need, void* stream) {
    if (need <= g_ws_cap[kind][dev][slot]) return g_ws_ptr[kind][dev][slot];
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing((cudaStream_t)stream, &cs);
    if (cs != cudaStreamCaptureStatusNone) return nullptr;
    const size_t cap = std::max<size_t>(need, (size_t)(kind ? 64 : 32) << 20);
    float* q = nullptr;
    if (cudaMalloc(&q, cap) != cudaSuccess) return nullptr;
    g_ws_ptr[kind][dev][slot] = q;
    g_ws_cap[kind][dev][slot] = cap;
    return q;
}
extern "C" float* mlb_workspace_get(int kind, size_t need, void* stream) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 64 || kind < 0 || kind > 1) return nullptr;
    std::lock_guard<std::mutex> lk(g_ws_mu);
    return ws_grow(kind, dev, g_ws_slot, need, stream);
}
// Give slots 1 .. n_slots-1 of the current device the capacity slot 0 has reached, so that work that moves to side
// streams INSIDE a stream capture (where nothing can be allocated) finds its workspace: call after an eager warm-up
// of the same code on one stream.
extern "C" int mlb_reserve_workspace_slots(int32_t n_slots) {
    if (n_slots < 1 || n_slots > MLB_WS_SLOTS) return MLB_EINVAL;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 64) return MLB_EINVAL;
    std::lock_guard<std::mutex> lk(g_ws_mu);
    for (int kind = 0; kind < 2; kind++)
        for (int s = 1; s < n_slots; s++)
            if (g_ws_cap[kind][dev][0] > g_ws_cap[kind][dev][s] && !ws_grow(kind, dev, s, g_ws_cap[kind][dev][0], nullptr))
                return MLB_ENOMEM;
    return MLB_OK;
}

extern "C" {

int mlb_gemm(const float* A, int64_t a_bs, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_bs,
             int64_t b_rs, int64_t b_cs, float* C, int64_t c_bs, int64_t ldc, const float* bias,
             int64_t bias_bs, int32_t M, int32_t N, int32_t K, int32_t batch, float beta, int32_t act,
             void* stream) {
    if (!A || !B || !C || M < 0 || N < 0 || K < 0 || batch < 1) return MLB_EINVAL;
    if (M == 0 || N == 0) return MLB_OK;
    // single products big enough to fill tensor-core tiles (>= 2^21 multiply-adds) go to the tcgen05 kernel
    // (csrc/mlb_gemm_tc.cu)
    if (batch == 1 && (int64_t)M * N * K >= ((int64_t)1 << 21) &&
        mlb_gemm_tc_supported(A, a_rs, a_cs, B, b_rs, b_cs, C, ldc, M, N, K)) {
        const int rc = mlb_gemm_tc(A, a_rs, a_cs, B, b_rs, b_cs, C, ldc, bias, M, N, K, beta, act, stream);
        if (rc != MLB_ESTATE && rc != MLB_ENOMEM) return rc;   // those two: nothing was launched, use the FFMA kernel
    }
    if (batch == 1 && K >= 1) {
        cudaStream_t st = (cudaStream_t)stream;
        if (K <= 8) {
            gemm_thin_k_kernel<<<nblk((int64_t)M * N, 256), 256, 0, st>>>(A, a_rs, a_cs, B, b_rs, b_cs, C, ldc, bias, M, N, K, beta, act);
            return ok();
        }
        if (N <= 8) {
            gemm_skinny_n_kernel<8><<<nblk((int64_t)M * 32, 128), 128, 0, st>>>(A, a_rs, a_cs, B, b_rs, b_cs, C, ldc, bias, M, N, K, beta, act);
            return ok();
        }
        if (M <= 8) {
            gemm_skinny_m_kernel<8><<<nblk(N, 32), dim3(32, 32), 0, st>>>(A, a_rs, a_cs, B, b_rs, b_cs, C, ldc, bias, M, N, K, beta, act);
            return ok();
        }
    }
    dim3 grid((N + BN - 1) / BN, (M + BM - 1) / BM, batch);
    // few output tiles and a long reduction: split K over more thread blocks (workspace per device, grown
    // outside stream capture only)
    int splits = 1;
    const int64_t tiles = (int64_t)grid.x * grid.y * batch;
    if (tiles < 64 && K >= 256) {
        splits = (int)std::min<int64_t>(std::min<int64_t>(16, 160 / tiles), K / 128);
        if (splits < 2) splits = 1;
    }
    float* ws = nullptr;
    if (splits > 1) {
        ws = mlb_workspace_get(0, (size_t)splits * batch * M * N * sizeof(float), stream);
        if (!ws) splits = 1;
    }
    grid.z = batch * splits;
    gemm_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(A, a_bs, a_rs, a_cs, B, b_bs, b_rs, b_cs, C, c_bs, ldc,
                                                        bias, bias_bs, M, N, K, beta, act, splits, ws);
    if (splits > 1)
        splitk_reduce_kernel<<<nblk((int64_t)M * N * batch, 256), 256, 0, (cudaStream_t)stream>>>(
            ws, splits, batch, C, c_bs, ldc, bias, bias_bs, M, N, beta, act);
    return ok();
}

int mlb_gru_gates_forward(const float* gi, const float* gh, const float* h, float* h_new, float* gates,
                          int32_t M, int32_t H, void* stream) {
    if (!gi || !gh || !h || !h_new) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    gru_gates_fwd_kernel<<<nblk((int64_t)M * H, 256), 256, 0, (cudaStream_t)stream>>>(gi, gh, h, h_new, gates, M, H);
    return ok();
}

int mlb_gru_gates_backward(const float* dh_new, const float* gates, const float* h, const float* gh,
                           float* dgi, float* dgh, float* dh_direct, int32_t M, int32_t H, void* stream) {
    if (!dh_new || !gates || !h || !gh || !dgi || !dgh || !dh_direct) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    gru_gates_bwd_kernel<<<nblk((int64_t)M * H, 256), 256, 0, (cudaStream_t)stream>>>(dh_new, gates, h, gh, dgi, dgh, dh_direct, M, H);
    return ok();
}

int mlb_relu_backward(const float* y, const float* dy, float* dx, int64_t n, void* stream) {
    if (!y || !dy || !dx) return MLB_EINVAL;
    if (n == 0) return MLB_OK;
    relu_bwd_kernel<<<nblk(n, 256), 256, 0, (cudaStream_t)stream>>>(y, dy, dx, n);
    return ok();
}

int mlb_abs_backward(const float* pre, const float* dy, float* dx, int64_t n, void* stream) {
    if (!pre || !dy || !dx) return MLB_EINVAL;
    if (n == 0) return MLB_OK;
    abs_bwd_kernel<<<nblk(n, 256), 256, 0, (cudaStream_t)stream>>>(pre, dy, dx, n);
    return ok();
}

int mlb_colsum(const float* dy, float* db, int32_t M, int32_t N, int64_t ld, float beta, void* stream) {
    if (!dy || !db) return MLB_EINVAL;
    if (N == 0) return MLB_OK;
    colsum_kernel<<<(N + 31) / 32, dim3(32, 32), 0, (cudaStream_t)stream>>>(dy, db, M, N, ld, beta);
    return ok();
}

int mlb_axpby(float a, const float* x, float b, float* y, int64_t n, void* stream) {
    if (!x || !y) return MLB_EINVAL;
    if (n == 0) return MLB_OK;
    axpby_kernel<<<nblk(n, 256), 256, 0, (cudaStream_t)stream>>>(a, x, b, y, n);
    return ok();
}

int mlb_sumsq(const float* x, int64_t n, double* out_accum, void* stream) {
    if (!x || !out_accum) return MLB_EINVAL;
    if (n == 0) return MLB_OK;
    unsigned blocks = nblk(n, 256);
    blocks = blocks > 1024 ? 1024 : blocks;
    sumsq_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, n, out_accum);
    return ok();
}

int mlb_scale(float* x, int64_t n, const double* norm_sq, float max_norm, void* stream) {
    if (!x || !norm_sq) return MLB_EINVAL;
    if (n == 0) return MLB_OK;
    scale_kernel<<<nblk(n, 256), 256, 0, (cudaStream_t)stream>>>(x, n, norm_sq, max_norm);
    return ok();
}

int mlb_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
             float eps, int32_t step, void* stream) {
    if (!p || !g || !m || !v || step < 1) return MLB_EINVAL;
    if (n == 0) return MLB_OK;
    const double bc1 = 1.0 - pow((double)beta1, (double)step);
    const double bc2 = 1.0 - pow((double)beta2, (double)step);
    adam_kernel<<<nblk(n, 256), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, beta1, beta2, eps,
                                                                (float)((double)lr / bc1), (float)sqrt(bc2));
    return ok();
}

int mlb_adam_dev(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                 float eps, int32_t* step_dev, float* coef_dev, void* stream) {
    if (!p || !g || !m || !v || !step_dev || !coef_dev) return MLB_EINVAL;
    adam_prep_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(step_dev, lr, beta1, beta2, coef_dev);
    if (n > 0)
        adam_dev_kernel<<<nblk(n, 256), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, beta1, beta2, eps, coef_dev);
    return ok();
}

int mlb_egreedy_select(const float* q, const float* u, const int32_t* rnd, float epsilon, int32_t* action,
                       float* q_sel, int32_t M, int32_t K, void* stream) {
    if (!q || !action || (u && !rnd) || K < 1) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    egreedy_kernel<<<nblk(M, 128), 128, 0, (cudaStream_t)stream>>>(q, u, rnd, epsilon, action, q_sel, M, K);
    return ok();
}

int mlb_onehot_action(const int32_t* action, int32_t M, int32_t Sa, int32_t stride, uint8_t hot, uint8_t cold,
                      uint8_t* out, void* stream) {
    if (!action || !out || Sa < 1) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    onehot_action_kernel<<<nblk((int64_t)M * Sa, 256), 256, 0, (cudaStream_t)stream>>>(action, M, Sa, stride, hot, cold, out);
    return ok();
}

int mlb_row_max(const float* q, float* out, int32_t* argmax, int32_t M, int32_t K, void* stream) {
    if (!q || !out || K < 1) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    row_max_kernel<<<nblk(M, 128), 128, 0, (cudaStream_t)stream>>>(q, out, argmax, M, K);
    return ok();
}

int mlb_mixer_forward(const float* q, const float* w1, const float* b1, const float* w2, const float* b2,
                      float* q_tot, float* hidden_out, int32_t M, int32_t A, int32_t E, void* stream) {
    if (!q || !w1 || !b1 || !w2 || !b2 || !q_tot) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    mixer_fwd_kernel<<<nblk((int64_t)M * 32, 128), 128, 0, (cudaStream_t)stream>>>(q, w1, b1, w2, b2, q_tot, hidden_out, M, A, E);
    return ok();
}

int mlb_mixer_backward(const float* dq_tot, const float* q, const float* w1, const float* w2, const float* hidden,
                       float* dq, float* dw1, float* db1, float* dw2, float* db2, int32_t M, int32_t A,
                       int32_t E, void* stream) {
    if (!dq_tot || !q || !w1 || !w2 || !hidden || !dq || !dw1 || !db1 || !dw2 || !db2) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    mixer_bwd_kernel<<<nblk((int64_t)M * 32, 128), 128, 0, (cudaStream_t)stream>>>(dq_tot, q, w1, w2, hidden, dq, dw1, db1, dw2, db2, M, A, E);
    return ok();
}

int mlb_tanh_gaussian_forward(const float* mean, const float* log_std_raw, const float* eps, float lo, float hi,
                              float scale, float bias, float* action, float* logp, float* mean_action,
                              int32_t M, int32_t A, void* stream) {
    if (!mean || !log_std_raw) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    tanh_gauss_fwd_kernel<<<nblk((int64_t)M * 32, 128), 128, 0, (cudaStream_t)stream>>>(mean, log_std_raw, eps, lo, hi, scale, bias,
                                                                                         action, logp, mean_action, M, A);
    return ok();
}

int mlb_tanh_gaussian_backward(const float* mean, const float* log_std_raw, const float* eps, float lo, float hi,
                               float scale, const float* d_action, const float* d_logp, float* d_mean,
                               float* d_log_std_raw, int32_t M, int32_t A, void* stream) {
    if (!mean || !log_std_raw || !eps || !d_mean || !d_log_std_raw) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    tanh_gauss_bwd_kernel<<<nblk((int64_t)M * A, 256), 256, 0, (cudaStream_t)stream>>>(mean, log_std_raw, eps, lo, hi, scale,
                                                                                       d_action, d_logp, d_mean, d_log_std_raw, M, A);
    return ok();
}

int mlb_abs_forward(const float* x, float* y, int64_t n, void* stream) {
    if (!x || !y) return MLB_EINVAL;
    if (n == 0) return MLB_OK;
    abs_fwd_kernel<<<nblk(n, 256), 256, 0, (cudaStream_t)stream>>>(x, y, n);
    return ok();
}

int mlb_qmix_td_loss(const float* q_tot, const float* target_q_tot, const float* reward_sum, const float* done,
                     const int32_t* seq_len, float gamma, float* targets, float* dq_tot, double* stats,
                     int32_t B, int32_t T, void* stream) {
    if (!q_tot || !target_q_tot || !reward_sum || !done || !seq_len || !targets || !dq_tot || !stats) return MLB_EINVAL;
    qmix_td_loss_kernel<<<1, 512, 0, (cudaStream_t)stream>>>(q_tot, target_q_tot, reward_sum, done, seq_len, gamma, targets, dq_tot, stats, B, T);
    return ok();
}

int mlb_sac_q_target(const float* reward, const float* done, const float* q1n, const float* q2n, const float* logp_next,
                     const float* alpha, float gamma, float* y, int32_t M, void* stream) {
    if (!reward || !done || !q1n || !q2n || !logp_next || !alpha || !y) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    sac_q_target_kernel<<<nblk(M, 256), 256, 0, (cudaStream_t)stream>>>(reward, done, q1n, q2n, logp_next, alpha, gamma, y, M);
    return ok();
}

int mlb_mse_loss(const float* q, const float* y, float* dq, double* loss, int32_t M, void* stream) {
    if (!q || !y || !dq || !loss || M < 1) return MLB_EINVAL;
    mse_loss_kernel<<<1, 512, 0, (cudaStream_t)stream>>>(q, y, dq, loss, M);
    return ok();
}

int mlb_sac_policy_loss(const float* logp, const float* q1, const float* q2, const float* alpha, float* d_logp,
                        float* dq1, float* dq2, double* loss, int32_t M, void* stream) {
    if (!logp || !q1 || !q2 || !alpha || !d_logp || !dq1 || !dq2 || !loss || M < 1) return MLB_EINVAL;
    sac_policy_loss_kernel<<<1, 512, 0, (cudaStream_t)stream>>>(logp, q1, q2, alpha, d_logp, dq1, dq2, loss, M);
    return ok();
}

int mlb_sac_alpha_loss(const float* logp, const float* log_alpha, float target_entropy, float* d_log_alpha,
                       double* loss, int32_t M, void* stream) {
    if (!logp || !log_alpha || !d_log_alpha || !loss || M < 1) return MLB_EINVAL;
    sac_alpha_loss_kernel<<<1, 512, 0, (cudaStream_t)stream>>>(logp, log_alpha, target_entropy, d_log_alpha, loss, M);
    return ok();
}

int mlb_exp_scalar(const float* x, float* y, void* stream) {
    if (!x || !y) return MLB_EINVAL;
    exp_scalar_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(x, y);
    return ok();
}

int mlb_softmax_forward(const float* x, float* y, int64_t rows, int32_t n, void* stream) {
    if (!x || !y || n < 1 || n > 64) return MLB_EINVAL;
    if (rows == 0) return MLB_OK;
    softmax_fwd_kernel<<<nblk(rows, 128), 128, 0, (cudaStream_t)stream>>>(x, y, rows, n);
    return ok();
}

int mlb_softmax_backward(const float* y, const float* dy, float* dx, int64_t rows, int32_t n, void* stream) {
    if (!y || !dy || !dx || n < 1 || n > 64) return MLB_EINVAL;
    if (rows == 0) return MLB_OK;
    softmax_bwd_kernel<<<nblk(rows, 128), 128, 0, (cudaStream_t)stream>>>(y, dy, dx, rows, n);
    return ok();
}

int mlb_concat_onehot(const float* x, const int32_t* action, float* out, int64_t rows, int32_t F, int32_t heads,
                      int32_t n, void* stream) {
    if (!x || !action || !out || F < 0 || heads < 1 || n < 1) return MLB_EINVAL;
    if (rows == 0) return MLB_OK;
    concat_onehot_kernel<<<nblk(rows * (F + heads * n), 256), 256, 0, (cudaStream_t)stream>>>(x, action, out, rows, F, heads, n);
    return ok();
}

int mlb_categorical(const float* p, const float* u, const int32_t* given, int32_t* action, float* logp, float* psel,
                    int64_t rows, int32_t n, void* stream) {
    if (!p || n < 1) return MLB_EINVAL;
    if (rows == 0) return MLB_OK;
    categorical_kernel<<<nblk(rows, 128), 128, 0, (cudaStream_t)stream>>>(p, u, given, action, logp, psel, rows, n);
    return ok();
}

int mlb_logprob_backward(const float* p, const int32_t* action, const float* g, float* dlogits, int64_t rows,
                         int32_t n, int32_t group, void* stream) {
    if (!p || !action || !g || !dlogits || n < 1 || group < 1) return MLB_EINVAL;
    if (rows == 0) return MLB_OK;
    logprob_bwd_kernel<<<nblk(rows * n, 256), 256, 0, (cudaStream_t)stream>>>(p, action, g, dlogits, rows, n, group);
    return ok();
}

int mlb_scatter_class(const float* g, const int32_t* action, float* d, int64_t rows, int32_t n, void* stream) {
    if (!g || !action || !d || n < 1) return MLB_EINVAL;
    if (rows == 0) return MLB_OK;
    scatter_class_kernel<<<nblk(rows * n, 256), 256, 0, (cudaStream_t)stream>>>(g, action, d, rows, n);
    return ok();
}

int mlb_weighted_sum_forward(const float* q, const float* w, float* out, int32_t M, int32_t A, void* stream) {
    if (!q || !w || !out || A < 1) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    weighted_sum_fwd_kernel<<<nblk(M, 128), 128, 0, (cudaStream_t)stream>>>(q, w, out, M, A);
    return ok();
}

int mlb_weighted_sum_backward(const float* g, const float* q, const float* w, float* dq, float* dw, int32_t M,
                              int32_t A, void* stream) {
    if (!g || !q || !w || !dq || !dw || A < 1) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    weighted_sum_bwd_kernel<<<nblk((int64_t)M * A, 256), 256, 0, (cudaStream_t)stream>>>(g, q, w, dq, dw, (int64_t)M * A, A);
    return ok();
}

int mlb_td_lambda_targets(const float* reward, const float* target_q, float* ret, float gamma, float td_lambda,
                          int32_t B, int32_t T, void* stream) {
    if (!reward || !target_q || !ret || B < 1 || T < 1) return MLB_EINVAL;
    td_lambda_kernel<<<nblk(B, 128), 128, 0, (cudaStream_t)stream>>>(reward, target_q, ret, gamma, td_lambda, B, T);
    return ok();
}

int mlb_reward_normalize(const float* reward, float* out, float scale, int32_t B, int32_t T, void* stream) {
    if (!reward || !out || B < 2 || T < 1) return MLB_EINVAL;
    reward_norm_kernel<<<nblk(T, 64), 64, 0, (cudaStream_t)stream>>>(reward, out, scale, B, T);
    return ok();
}

int mlb_dsac_q_target(const float* reward, const float* q1n, const float* q2n, const float* logp_next,
                      const float* alpha, float gamma, float* y, int32_t M, void* stream) {
    if (!reward || !q1n || !q2n || !logp_next || !alpha || !y) return MLB_EINVAL;
    if (M == 0) return MLB_OK;
    dsac_q_target_kernel<<<nblk(M, 256), 256, 0, (cudaStream_t)stream>>>(reward, q1n, q2n, logp_next, alpha, gamma, y, M);
    return ok();
}

int mlb_replay_push(const float* state, const float* action, const double* reward, const float* next_state,
                    const uint8_t* done, const float* hidden, float* r_state, float* r_action, float* r_reward,
                    float* r_next_state, float* r_done, float* r_hidden, int64_t* pos_dev, int32_t n, int32_t capacity,
                    int32_t state_dim, int32_t action_dim, int32_t hidden_dim, void* stream) {
    if (!state || !action || !reward || !next_state || !done || !hidden || !r_state || !r_action || !r_reward ||
        !r_next_state || !r_done || !r_hidden || !pos_dev || n < 0 || n > capacity)
        return MLB_EINVAL;
    if (n == 0) return MLB_OK;
    ReplayPtrs r{r_state, r_action, r_next_state, r_hidden, r_reward, r_done};
    replay_push_kernel<<<n, 256, 0, (cudaStream_t)stream>>>(state, action, reward, next_state, done, hidden, r, pos_dev,
                                                          capacity, state_dim, action_dim, hidden_dim);
    replay_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(pos_dev, n, capacity);
    return ok();
}

int mlb_replay_gather(const float* r_state, const float* r_action, const float* r_reward, const float* r_next_state,
                      const float* r_done, const float* r_hidden, const int64_t* idx, float* state, float* action,
                      float* reward, float* next_state, float* done, float* hidden, int32_t batch, int32_t state_dim,
                      int32_t action_dim, int32_t hidden_dim, void* stream) {
    if (!r_state || !r_action || !r_reward || !r_next_state || !r_done || !r_hidden || !idx || !state || !action ||
        !reward || !next_state || !done || !hidden || batch < 0)
        return MLB_EINVAL;
    if (batch == 0) return MLB_OK;
    ReplayPtrs r{const_cast<float*>(r_state), const_cast<float*>(r_action), const_cast<float*>(r_next_state),
                 const_cast<float*>(r_hidden), const_cast<float*>(r_reward), const_cast<float*>(r_done)};
    replay_gather_kernel<<<batch, 256, 0, (cudaStream_t)stream>>>(r, idx, state, action, reward, next_state, done, hidden,
                                                                state_dim, action_dim, hidden_dim);
    return ok();
}

int mlb_gru_seq_forward(const float* gi_all, const float* W_hh, const float* b_hh, const float* h0, float* hs,
                        float* hprev, float* ghs, float* gates, int32_t T, int32_t B, int32_t H, void* stream) {
    if (!gi_all || !W_hh || !b_hh || !h0 || !hs || T < 0 || B < 0 || H < 1) return MLB_EINVAL;
    if (T == 0 || B == 0) return MLB_OK;
    const size_t smem = ((size_t)(3 * H + 1) * H + (size_t)GRU_SEQ_RB * H + (size_t)GRU_SEQ_RB * 3 * H) * sizeof(float);
    if (3 * H > 1024 || smem > 227 * 1024) return MLB_EINVAL;
    if (cudaFuncSetAttribute(gru_seq_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return MLB_ECUDA;
    gru_seq_fwd_kernel<<<(B + GRU_SEQ_RB - 1) / GRU_SEQ_RB, 3 * H, smem, (cudaStream_t)stream>>>(gi_all, W_hh, b_hh, h0, hs, hprev, ghs,
                                                                                          gates, T, B, H);
    return ok();
}

int mlb_gru_seq_backward(const float* dhs, const float* gates, const float* hprev, const float* ghs, const float* W_hh,
                         float* dgi_all, float* dgh_all, float* dh0, int32_t T, int32_t B, int32_t H, void* stream) {
    if (!dhs || !gates || !hprev || !ghs || !W_hh || !dgi_all || !dgh_all || T < 0 || B < 0 || H < 1) return MLB_EINVAL;
    if (T == 0 || B == 0) return MLB_OK;
    const size_t smem = ((size_t)3 * H * H + (size_t)GRU_SEQ_RB * H + (size_t)GRU_SEQ_RB * 3 * H + (size_t)3 * GRU_SEQ_RB * H) * sizeof(float);
    if (3 * H > 1024 || smem > 227 * 1024) return MLB_EINVAL;
    if (cudaFuncSetAttribute(gru_seq_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return MLB_ECUDA;
    gru_seq_bwd_kernel<<<(B + GRU_SEQ_RB - 1) / GRU_SEQ_RB, 3 * H, smem, (cudaStream_t)stream>>>(dhs, gates, hprev, ghs, W_hh, dgi_all,
                                                                                          dgh_all, dh0, T, B, H);
    return ok();
}

}  // extern "C"
