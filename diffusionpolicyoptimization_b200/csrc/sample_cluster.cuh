// Persistent small-batch DDPM chain sampler (VPGDiffusion.call, diffusion_vpg.py:249-339).
//
// ONE launch per rollout step; all T denoising steps loop on-chip.  The grid is a set of 16-CTA
// thread-block clusters (one per GPC: 8 x 16 = 128 of the 148 SMs - a GPC hosts one 16-CTA cluster).  A cluster owns R env rows
// for the whole chain; inside a cluster every CTA owns 32 of the 512 hidden columns:
//   * its [512 x 32] fp32 slice of block.l1 stays resident in shared memory (reloaded once at the base -> fine-tuned switch, t = K-1);
//   * no activation sits between block.l2 and the output layer (model/common/mlp.py ResidualMLP + final Dense), so
//       eps = (relu(h1) W2 + b2 + u) W3 + b3 = relu(h1) (W2 W3) + u W3 + (b2 W3 + b3):
//     the CTA keeps its 32 rows of W23 = W2 W3 (folded per weight version, double accumulation) and of W3 and never forms v -
//     the second H x H product AND its exchange (all-gather of relu(h1) + cluster barrier) disappear from the chain;
//   * its 512 threads each keep one column of the layer-0 x-rows (W_in[0:A, c]) and the
//     obs contribution  obs @ W_in[A+td:, c]  in registers (the obs term is constant over the chain);
//   * the time embedding enters as a per-t bias row bt[t] (precomputed per weight version).
// Per denoising step: L0 (every CTA all 512 columns: 120 FMAs per thread, cheaper than an exchange) -> L1 slice (K split over the
// 16 warps, shared-memory reduction) -> partial eps over the CTA's 32 columns, written straight into the 16 CTAs' buffers (DSMEM)
// -> cluster barrier -> posterior / noise / x update (redundant, bit-identical in all 16 CTAs).  ONE cluster barrier and four block
// barriers per step; the next step's bias row and this step's noise are fetched before the exchange.
// Strict fp32 FFMA; noise is injected (parity) or drawn in-kernel by Philox4x32-10.
// Measured and dropped (round 2): splitting K over the lanes of a warp with a butterfly instead of over the warps (126 -> 145 us per
// 40-env rollout step: 120 extra shuffle / add instructions per thread and layer); scattering 8-byte pairs to the 16 CTAs without
// staging (165 us: 16 small DSMEM packets per store instead of one 128-byte row segment).
#pragma once
#include "simt_kernels.cuh"
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

constexpr int CS_H = 512;        // hidden width this kernel is specialised for
constexpr int CS_C = 16;         // CTAs per cluster
constexpr int CS_COLS = CS_H / CS_C;   // 32 hidden columns per CTA
constexpr int CS_THREADS = 512;

struct ClusterSampleP {
    const float* w[2];        // flat actor parameters: [0] base, [1] fine-tuned
    const float* bt[2];       // per-t layer-0 bias rows [T][H]
    const float* w23[2];      // folded output layer W2 @ W3 [H][A]
    const float* b23[2];      // b2 @ W3 + b3 [A]
    ActorOff o;
    const float* obs; const float* xT; const float* noise;
    float* actions; float* chains;
    const float* sch;
    int B, A, Do, T, K, td, nchunks, use_base_policy;
    SampleHyper hp;
    uint64_t seed, offset; int64_t row_offset;
    // env-side epilogue (SURVEY.md 8f.4): the first act_cols = act_steps * Da entries of every action chunk, un-normalised like
    // MujocoLocomotionLowdimWrapper.unnormalize_action, written where the env workers read them (pinned host memory or device)
    float* raw_actions; const float* act_min; const float* act_max; int act_cols, Da;
};
// env/gym_utils/wrapper/mujoco_locomotion_lowdim.py:60-62 in NumPy's fp32 evaluation order (no FMA contraction)
__device__ __forceinline__ float env_unnormalize_action(float a, float amin, float amax) {
    const float a01 = __fdiv_rn(__fadd_rn(a, 1.f), 2.f);
    return __fadd_rn(__fmul_rn(a01, __fsub_rn(amax, amin)), amin);
}

template <int AP, int R>
constexpr size_t cluster_sample_smem_floats() {
    return (size_t)CS_H * CS_COLS          // W1s
         + (size_t)2 * CS_COLS * AP        // W3s, W23s
         + (size_t)2 * R * CS_H            // actA, red
         + (size_t)2 * R * CS_COLS         // uown, out1
         + (size_t)R * AP * (1 + 2 * CS_C) // xs, part[2][16]
         + CS_COLS + AP;                   // b1s, b3s
}

template <int AP, int R>
__global__ void __launch_bounds__(CS_THREADS, 1) sample_cluster_kernel(const ClusterSampleP p) {
    cg::cluster_group cluster = cg::this_cluster();
    const int crank = (int)cluster.block_rank();
    const int cid = blockIdx.x / CS_C, nclusters = gridDim.x / CS_C;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int col0 = crank * CS_COLS;
    const int A = p.A, T = p.T, K = p.K, B = p.B;

    extern __shared__ __align__(16) float smem[];
    float* W1s = smem;                         // [512][32]
    float* W3s = W1s + CS_H * CS_COLS;         // [32][AP]  rows col0.. of W3 (the residual's path to eps)
    float* W23s = W3s + CS_COLS * AP;          // [32][AP]  rows col0.. of W2 @ W3
    float* actA = W23s + CS_COLS * AP;         // [R][512] relu(u)
    float* red = actA + R * CS_H;              // [16][R][32] cross-warp partials
    float* uown = red + R * CS_H;              // [R][32] raw u, own columns (residual)
    float* out1 = uown + R * CS_COLS;          // [R][32] relu(h1), own columns
    float* xs = out1 + R * CS_COLS;            // [R][AP] current x
    float* part = xs + R * AP;                 // [2][16][R][AP] partial eps of every CTA; two buffers by step parity: with ONE cluster
                                               // barrier per step a fast CTA may already send step i + 1 while a slow one still sums step i
    float* b1s = part + 2 * CS_C * R * AP;     // [32]
    float* b3s = b1s + CS_COLS;                // [AP]  b2 @ W3 + b3

    float wx[AP];        // W_in[a][tid]
    float cobs[R];       // obs[r] @ W_in[A+td:, tid]

    for (int chunk = cid; chunk < p.nchunks; chunk += nclusters) {
        const int row0 = chunk * R;
        // ---- initialise x (x_T injected or Philox slot 0)
        if (tid < R * AP) {
            int r = tid / AP, a = tid % AP;
            float v = 0.f;
            if (a < A && row0 + r < B) {
                v = p.xT ? p.xT[(size_t)(row0 + r) * A + a]
                         : philox_normal(p.seed, p.offset, p.row_offset + row0 + r, 0, a);
                if (crank == 0 && p.chains && K == T) p.chains[((size_t)(row0 + r) * (K + 1)) * A + a] = v;
            }
            xs[tid] = v;
        }
        __syncthreads();
        int cur_net = -1;
        float bt_pref = 0.f;       // bt[t][tid] of the coming step, fetched one step ahead: its L2 latency hides behind the two products

        for (int i = 0; i < T; ++i) {
            const int t = T - 1 - i;
            const int net = (t < K && !p.use_base_policy) ? 1 : 0;
            float btv = bt_pref;
            if (net != cur_net) {
                // ---- (re)load this net's resident slices and recompute its obs term
                const float* w = p.w[net];
                btv = p.bt[net][(size_t)t * CS_H + tid];
                for (int idx = tid; idx < CS_H * CS_COLS; idx += CS_THREADS) {
                    int k = idx >> 5, j = idx & 31;
                    W1s[idx] = w[p.o.w1 + (size_t)k * CS_H + col0 + j];
                }
                for (int idx = tid; idx < CS_COLS * AP; idx += CS_THREADS) {
                    int k = idx / AP, a = idx % AP;
                    W3s[idx] = a < A ? w[p.o.w3 + (size_t)(col0 + k) * A + a] : 0.f;
                    W23s[idx] = a < A ? p.w23[net][(size_t)(col0 + k) * A + a] : 0.f;
                }
                if (tid < CS_COLS) b1s[tid] = w[p.o.b1 + col0 + tid];
                if (tid < AP) b3s[tid] = tid < A ? p.b23[net][tid] : 0.f;
#pragma unroll
                for (int a = 0; a < AP; ++a) wx[a] = a < A ? w[p.o.win + (size_t)a * CS_H + tid] : 0.f;
#pragma unroll
                for (int r = 0; r < R; ++r) cobs[r] = 0.f;
                for (int j = 0; j < p.Do; ++j) {
                    float wv = w[p.o.win + (size_t)(A + p.td + j) * CS_H + tid];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        float ov = (row0 + r < B) ? p.obs[(size_t)(row0 + r) * p.Do + j] : 0.f;
                        cobs[r] = fmaf(ov, wv, cobs[r]);
                    }
                }
                cur_net = net;
                __syncthreads();
            }
            // ---- L0 (every CTA computes all 512 columns): u = [x|obs] @ W_in + bt[t]
            {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    float u = cobs[r] + btv;
#pragma unroll
                    for (int a = 0; a < AP; ++a) u = fmaf(xs[r * AP + a], wx[a], u);
                    actA[r * CS_H + tid] = fmaxf(u, 0.f);
                    if (tid >= col0 && tid < col0 + CS_COLS) uown[r * CS_COLS + tid - col0] = u;
                }
                if (i + 1 < T) {
                    const int t1 = t - 1, net1 = (t1 < K && !p.use_base_policy) ? 1 : 0;
                    bt_pref = p.bt[net1][(size_t)t1 * CS_H + tid];
                }
            }
            // this step's noise does not depend on eps: fetch / draw it before the exchanges
            float nz = 0.f;
            if (tid < R * AP) {
                const int r = tid / AP, a = tid % AP;
                if (a < A && row0 + r < B) {
                    const int64_t row = row0 + r;
                    nz = p.noise ? p.noise[((size_t)i * B + row) * A + a] : philox_normal(p.seed, p.offset, p.row_offset + row, 1 + i, a);
                }
            }
            __syncthreads();
            // ---- L1 slice: h1[:, col0:col0+32] = relu(u) @ W1[:, cols] + b1
            {
                float acc[R];
#pragma unroll
                for (int r = 0; r < R; ++r) acc[r] = 0.f;
                const float* Wp = W1s + (warp * 32) * CS_COLS + lane;
                const float* ap = actA + warp * 32;
#pragma unroll
                for (int kk = 0; kk < 32; kk += 4) {
                    float w0 = Wp[(kk + 0) * CS_COLS], w1 = Wp[(kk + 1) * CS_COLS];
                    float w2 = Wp[(kk + 2) * CS_COLS], w3 = Wp[(kk + 3) * CS_COLS];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        float4 a = *reinterpret_cast<const float4*>(ap + r * CS_H + kk);
                        acc[r] = fmaf(a.x, w0, acc[r]); acc[r] = fmaf(a.y, w1, acc[r]);
                        acc[r] = fmaf(a.z, w2, acc[r]); acc[r] = fmaf(a.w, w3, acc[r]);
                    }
                }
#pragma unroll
                for (int r = 0; r < R; ++r) red[(warp * R + r) * 32 + lane] = acc[r];
            }
            __syncthreads();
            if (tid < R * 32) {
                int r = tid >> 5;
                float s = b1s[lane];
#pragma unroll
                for (int w = 0; w < 16; ++w) s += red[(w * R + r) * 32 + lane];
                out1[r * 32 + lane] = fmaxf(s, 0.f);
            }
            __syncthreads();
            // ---- partial output layer over this CTA's 32 columns, written straight into the 16 CTAs' partial buffers (contiguous per warp)
            if (tid < R * AP) {
                int r = tid / AP, a = tid % AP;
                float s = 0.f;
#pragma unroll
                for (int k = 0; k < CS_COLS; ++k) s = fmaf(out1[r * 32 + k], W23s[k * AP + a], s);
                float s2 = 0.f;
#pragma unroll
                for (int k = 0; k < CS_COLS; ++k) s2 = fmaf(uown[r * 32 + k], W3s[k * AP + a], s2);
                s += s2;
#pragma unroll
                for (int dst = 0; dst < CS_C; ++dst) cluster.map_shared_rank(part, dst)[((i & 1) * CS_C + crank) * (R * AP) + tid] = s;
            }
            cluster.sync();
            // ---- posterior mean / clipped noise / x update (identical in all 16 CTAs)
            if (tid < R * AP) {
                int r = tid / AP, a = tid % AP;
                if (a < A && row0 + r < B) {
                    float e = b3s[a];
#pragma unroll
                    for (int src = 0; src < CS_C; ++src) e += part[((i & 1) * CS_C + src) * (R * AP) + tid];
                    const int64_t row = row0 + r;
                    float xn = ddpm_step_elem(xs[tid], e, nz, t, p.sch, T, p.hp, t == 0);
                    xs[tid] = xn;
                    if (crank == 0) {
                        if (p.chains && t <= K) p.chains[((size_t)row * (K + 1) + (K - t)) * A + a] = xn;
                        if (t == 0) {
                            p.actions[(size_t)row * A + a] = xn;
                            if (p.raw_actions && a < p.act_cols)
                                p.raw_actions[(size_t)row * p.act_cols + a] = env_unnormalize_action(xn, p.act_min[a % p.Da], p.act_max[a % p.Da]);
                        }
                    }
                }
            }
            __syncthreads();
        }
    }
    // no CTA may exit while peers can still write into its shared memory
    cluster.sync();
}

// ---- wide chunks (32 < A <= 128): sample_cluster_wide_kernel<AP, R>, AP in {64, 128}
// The narrow kernel's layer 0 keeps one column of W_in's x-rows per thread (wx[AP]) and computes all 512 columns in every CTA.  At
// AP = 128 that column no longer fits the 128 registers a thread has at 512 threads, and the x-rows of all 512 columns (256 KB) do
// not fit shared memory either.  So here each CTA computes only its own 32 columns of u = [x|obs] @ W_in + bt[t]: its [AP][32]
// slice of the x-rows and the obs term of its columns stay resident, the K = AP product is split over the 16 warps like the L1
// slice, and relu(u) is all-gathered into every CTA's actA over DSMEM behind a second cluster barrier.  The rest of the step (L1
// slice, partial folded output layer, posterior update) is the narrow kernel's, with the (row, a) phases looping over R * AP > 512.
// Those phases are written out again rather than shared through helpers: moved into __device__ functions they changed the narrow
// kernel's generated code, and the A <= 32 instantiations are kept instruction for instruction.  A fix to one copy belongs in both.
// Two cluster barriers per step make ONE partial-eps buffer enough: a CTA writes step i + 1's partials only after the all-gather
// barrier of step i + 1, and every CTA arrives there after summing step i's.  Likewise peers write step i + 1's relu(u) into actA
// only after step i's partial barrier, which every CTA reaches after its L1 slice has read actA.
template <int AP, int R>
constexpr size_t cluster_sample_wide_smem_floats() {
    return (size_t)CS_H * CS_COLS          // W1s
         + (size_t)3 * CS_COLS * AP        // W3s, W23s, Wxs
         + (size_t)2 * R * CS_H            // actA, red
         + (size_t)3 * R * CS_COLS         // cobs, uown, out1
         + (size_t)R * AP * (1 + CS_C)     // xs, part[16]
         + CS_COLS + AP;                   // b1s, b3s
}

template <int AP, int R>
__global__ void __launch_bounds__(CS_THREADS, 1) sample_cluster_wide_kernel(const ClusterSampleP p) {
    static_assert(AP % 16 == 0 && AP > 32, "the x-rows of W_in are split evenly over the 16 warps");
    constexpr int NE = (R * AP + CS_THREADS - 1) / CS_THREADS;   // (row, a) elements per thread
    constexpr int KW = AP / 16;                                   // x-rows of W_in per warp in layer 0
    cg::cluster_group cluster = cg::this_cluster();
    const int crank = (int)cluster.block_rank();
    const int cid = blockIdx.x / CS_C, nclusters = gridDim.x / CS_C;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int col0 = crank * CS_COLS;
    const int A = p.A, T = p.T, K = p.K, B = p.B;

    extern __shared__ __align__(16) float smem[];
    float* W1s = smem;                         // [512][32]
    float* W3s = W1s + CS_H * CS_COLS;         // [32][AP]
    float* W23s = W3s + CS_COLS * AP;          // [32][AP]
    float* Wxs = W23s + CS_COLS * AP;          // [AP][32]  W_in[a][col0 + j], rows a >= A zeroed
    float* actA = Wxs + AP * CS_COLS;          // [R][512]  relu(u), all-gathered
    float* red = actA + R * CS_H;              // [16][R][32] cross-warp partials (layer 0, then L1)
    float* cobs = red + R * CS_H;              // [R][32]   obs[r] @ W_in[A+td:, col0 + j]
    float* uown = cobs + R * CS_COLS;          // [R][32]   raw u, own columns (residual)
    float* out1 = uown + R * CS_COLS;          // [R][32]   relu(h1), own columns
    float* xs = out1 + R * CS_COLS;            // [R][AP]   current x
    float* part = xs + R * AP;                 // [16][R][AP] partial eps of every CTA
    float* b1s = part + CS_C * R * AP;         // [32]
    float* b3s = b1s + CS_COLS;                // [AP]

    for (int chunk = cid; chunk < p.nchunks; chunk += nclusters) {
        const int row0 = chunk * R;
        // ---- initialise x (x_T injected or Philox slot 0)
#pragma unroll
        for (int q = 0; q < NE; ++q) {
            const int e = tid + q * CS_THREADS;
            if (e < R * AP) {
                const int r = e / AP, a = e % AP;
                float v = 0.f;
                if (a < A && row0 + r < B) {
                    v = p.xT ? p.xT[(size_t)(row0 + r) * A + a]
                             : philox_normal(p.seed, p.offset, p.row_offset + row0 + r, 0, a);
                    if (crank == 0 && p.chains && K == T) p.chains[((size_t)(row0 + r) * (K + 1)) * A + a] = v;
                }
                xs[e] = v;
            }
        }
        __syncthreads();
        int cur_net = -1;

        for (int i = 0; i < T; ++i) {
            const int t = T - 1 - i;
            const int net = (t < K && !p.use_base_policy) ? 1 : 0;
            if (net != cur_net) {
                // ---- (re)load this net's resident slices and recompute its obs term
                const float* w = p.w[net];
                for (int idx = tid; idx < CS_H * CS_COLS; idx += CS_THREADS) {
                    int k = idx >> 5, j = idx & 31;
                    W1s[idx] = w[p.o.w1 + (size_t)k * CS_H + col0 + j];
                }
                for (int idx = tid; idx < CS_COLS * AP; idx += CS_THREADS) {
                    int k = idx / AP, a = idx % AP;
                    W3s[idx] = a < A ? w[p.o.w3 + (size_t)(col0 + k) * A + a] : 0.f;
                    W23s[idx] = a < A ? p.w23[net][(size_t)(col0 + k) * A + a] : 0.f;
                }
                if (tid < CS_COLS) b1s[tid] = w[p.o.b1 + col0 + tid];
                if (tid < AP) b3s[tid] = tid < A ? p.b23[net][tid] : 0.f;
                for (int idx = tid; idx < AP * CS_COLS; idx += CS_THREADS) {
                    const int a = idx >> 5, j = idx & 31;
                    Wxs[idx] = a < A ? w[p.o.win + (size_t)a * CS_H + col0 + j] : 0.f;
                }
                if (tid < R * CS_COLS) {
                    const int r = tid >> 5;
                    float c = 0.f;
                    for (int j = 0; j < p.Do; ++j) {
                        const float ov = (row0 + r < B) ? p.obs[(size_t)(row0 + r) * p.Do + j] : 0.f;
                        c = fmaf(ov, w[p.o.win + (size_t)(A + p.td + j) * CS_H + col0 + lane], c);
                    }
                    cobs[tid] = c;
                }
                cur_net = net;
                __syncthreads();
            }
            // the bias row of this step's own columns and this step's noise do not depend on the products: fetch them first
            const float btv = tid < R * CS_COLS ? p.bt[net][(size_t)t * CS_H + col0 + lane] : 0.f;
            float nz[NE];
#pragma unroll
            for (int q = 0; q < NE; ++q) {
                const int e = tid + q * CS_THREADS;
                nz[q] = 0.f;
                if (e < R * AP) {
                    const int r = e / AP, a = e % AP;
                    if (a < A && row0 + r < B) {
                        const int64_t row = row0 + r;
                        nz[q] = p.noise ? p.noise[((size_t)i * B + row) * A + a] : philox_normal(p.seed, p.offset, p.row_offset + row, 1 + i, a);
                    }
                }
            }
            // ---- L0, own columns: u[:, col0:col0+32] = x @ W_in[0:AP, cols] (K split over the warps) + obs term + bt[t]
            {
                float acc[R];
#pragma unroll
                for (int r = 0; r < R; ++r) acc[r] = 0.f;
#pragma unroll
                for (int kk = 0; kk < KW; ++kk) {
                    const int a = warp * KW + kk;
                    const float wv = Wxs[a * CS_COLS + lane];
#pragma unroll
                    for (int r = 0; r < R; ++r) acc[r] = fmaf(xs[r * AP + a], wv, acc[r]);
                }
#pragma unroll
                for (int r = 0; r < R; ++r) red[(warp * R + r) * 32 + lane] = acc[r];
            }
            __syncthreads();
            if (tid < R * CS_COLS) {
                const int r = tid >> 5;
                float u = cobs[tid] + btv;
#pragma unroll
                for (int w = 0; w < 16; ++w) u += red[(w * R + r) * 32 + lane];
                uown[tid] = u;
                const float v = fmaxf(u, 0.f);
#pragma unroll 1
                for (int dst = 0; dst < CS_C; ++dst) cluster.map_shared_rank(actA, dst)[r * CS_H + col0 + lane] = v;
            }
            cluster.sync();    // relu(u) of all 512 columns is in every CTA's actA
            // ---- L1 slice: h1[:, col0:col0+32] = relu(u) @ W1[:, cols] + b1 (as in the narrow kernel)
            {
                float acc[R];
#pragma unroll
                for (int r = 0; r < R; ++r) acc[r] = 0.f;
                const float* Wp = W1s + (warp * 32) * CS_COLS + lane;
                const float* ap = actA + warp * 32;
#pragma unroll
                for (int kk = 0; kk < 32; kk += 4) {
                    float w0 = Wp[(kk + 0) * CS_COLS], w1 = Wp[(kk + 1) * CS_COLS];
                    float w2 = Wp[(kk + 2) * CS_COLS], w3 = Wp[(kk + 3) * CS_COLS];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        float4 a = *reinterpret_cast<const float4*>(ap + r * CS_H + kk);
                        acc[r] = fmaf(a.x, w0, acc[r]); acc[r] = fmaf(a.y, w1, acc[r]);
                        acc[r] = fmaf(a.z, w2, acc[r]); acc[r] = fmaf(a.w, w3, acc[r]);
                    }
                }
#pragma unroll
                for (int r = 0; r < R; ++r) red[(warp * R + r) * 32 + lane] = acc[r];
            }
            __syncthreads();
            if (tid < R * 32) {
                int r = tid >> 5;
                float s = b1s[lane];
#pragma unroll
                for (int w = 0; w < 16; ++w) s += red[(w * R + r) * 32 + lane];
                out1[r * 32 + lane] = fmaxf(s, 0.f);
            }
            __syncthreads();
            // ---- partial output layer over this CTA's 32 columns, written straight into the 16 CTAs' partial buffers
#pragma unroll
            for (int q = 0; q < NE; ++q) {
                const int e = tid + q * CS_THREADS;
                if (e < R * AP) {
                    const int r = e / AP, a = e % AP;
                    float s = 0.f;
#pragma unroll
                    for (int k = 0; k < CS_COLS; ++k) s = fmaf(out1[r * 32 + k], W23s[k * AP + a], s);
                    float s2 = 0.f;
#pragma unroll
                    for (int k = 0; k < CS_COLS; ++k) s2 = fmaf(uown[r * 32 + k], W3s[k * AP + a], s2);
                    s += s2;
#pragma unroll 1
                    for (int dst = 0; dst < CS_C; ++dst) cluster.map_shared_rank(part, dst)[crank * (R * AP) + e] = s;
                }
            }
            cluster.sync();
            // ---- posterior mean / clipped noise / x update (identical in all 16 CTAs)
#pragma unroll
            for (int q = 0; q < NE; ++q) {
                const int e = tid + q * CS_THREADS;
                if (e < R * AP) {
                    const int r = e / AP, a = e % AP;
                    if (a < A && row0 + r < B) {
                        float ev = b3s[a];
#pragma unroll
                        for (int src = 0; src < CS_C; ++src) ev += part[src * (R * AP) + e];
                        const int64_t row = row0 + r;
                        const float xn = ddpm_step_elem(xs[e], ev, nz[q], t, p.sch, T, p.hp, t == 0);
                        xs[e] = xn;
                        if (crank == 0) {
                            if (p.chains && t <= K) p.chains[((size_t)row * (K + 1) + (K - t)) * A + a] = xn;
                            if (t == 0) {
                                p.actions[(size_t)row * A + a] = xn;
                                if (p.raw_actions && a < p.act_cols)
                                    p.raw_actions[(size_t)row * p.act_cols + a] = env_unnormalize_action(xn, p.act_min[a % p.Da], p.act_max[a % p.Da]);
                            }
                        }
                    }
                }
            }
            __syncthreads();
        }
    }
    // no CTA may exit while peers can still write into its shared memory
    cluster.sync();
}

// ---- other hidden widths: sample_cluster_width_kernel<H, AP, R>, H in {256, 768, 1024}, AP in {32, 64, 128}
// The wide kernel's scheme for every chunk width: each CTA computes its own COLS = H / 16 columns of layer 0 from a resident
// [AP][COLS] slice of W_in's x-rows, relu(u) is all-gathered over DSMEM behind a cluster barrier, then the L1 slice, the partial
// folded output layer and the posterior update follow as in the wide kernel.  What changes with COLS:
//   * products over COLS columns (layer 0 and the L1 slice): lane & 15 picks a column, the thread owns the NC = COLS / 16 columns
//     c, c + 16, ... and lane >> 4 picks half of the R rows.  The two half-warps read the same weight address (broadcast) and two
//     relu(u) rows; actA rows are padded by 4 floats so those two float4 reads fall in different banks.  The K rows are split over
//     the 16 warps (H / 16 rows each) and reduced across warps in shared memory, as at H = 512;
//   * the W1 slice is partly resident: of each warp's H / 16 k-rows the first KRW stay in shared memory and the rest are read
//     from L2 (coalesced, one 64-byte segment per column group and half-warp) every denoising step.  KRW is the largest multiple
//     of 4 that the (H, AP, R) plan leaves room for (ClusterWidthPlan).  Which rows are resident does not change the order of
//     the sums, so the results do not depend on R.
// The H = 512 kernels above are left as they are (their A <= 32 and A > 32 instantiations keep their code instruction for
// instruction); a fix to the shared phases belongs in all three.
constexpr size_t CS_SMEM_FLOATS = 227 * 1024 / sizeof(float);   // the most dynamic shared memory a block can have (sm_100)

template <int H, int AP, int R>
struct ClusterWidthPlan {
    static constexpr int COLS = H / CS_C;
    static constexpr size_t fixed = (size_t)3 * COLS * AP          // W3s, W23s, Wxs
                                  + (size_t)R * (H + 4) + (size_t)R * H   // actA (rows padded by 4), red
                                  + (size_t)3 * R * COLS           // cobs, uown, out1
                                  + (size_t)R * AP * (1 + CS_C)    // xs, part[16]
                                  + COLS + AP;                     // b1s, b3s
    static constexpr bool fits = fixed <= CS_SMEM_FLOATS;
    // resident k-rows of W1 per warp: what is left, in multiples of 4, at most the warp's H / 16
    static constexpr size_t room = fits ? (CS_SMEM_FLOATS - fixed) / ((size_t)CS_C * COLS) / 4 * 4 : 0;
    static constexpr int krw = room < (size_t)(H / CS_C) ? (int)room : H / CS_C;
    static constexpr size_t floats = fixed + (size_t)krw * CS_C * COLS;
};
// the most rows per cluster pass whose plan fits
template <int H, int AP>
constexpr int cluster_width_rmax() {
    return ClusterWidthPlan<H, AP, 8>::fits ? 8 : ClusterWidthPlan<H, AP, 6>::fits ? 6 : ClusterWidthPlan<H, AP, 4>::fits ? 4 : 2;
}

template <int H, int AP, int R>
__global__ void __launch_bounds__(CS_THREADS, 1) sample_cluster_width_kernel(const ClusterSampleP p) {
    constexpr int COLS = H / CS_C;          // hidden columns per CTA
    constexpr int NC = COLS / 16;           // columns per thread in the products
    constexpr int RH = R / 2;               // rows per half-warp
    constexpr int LDA = H + 4;              // actA row stride
    constexpr int KPW = H / CS_C;           // k-rows of W1 per warp
    constexpr int KRW = ClusterWidthPlan<H, AP, R>::krw;   // of which resident
    constexpr int KW = AP / 16;             // x-rows of W_in per warp in layer 0
    constexpr int NE = (R * AP + CS_THREADS - 1) / CS_THREADS;
    static_assert(H % 256 == 0 && H != CS_H && H <= 1024, "widths other than 512, multiples of 256");
    static_assert(AP % 16 == 0 && R % 2 == 0 && R * COLS <= CS_THREADS, "thread mapping");
    static_assert(ClusterWidthPlan<H, AP, R>::fits && KRW % 4 == 0 && ClusterWidthPlan<H, AP, R>::floats <= CS_SMEM_FLOATS,
                  "shared-memory plan exceeds 227 KB");
    cg::cluster_group cluster = cg::this_cluster();
    const int crank = (int)cluster.block_rank();
    const int cid = blockIdx.x / CS_C, nclusters = gridDim.x / CS_C;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int c16 = lane & 15, half = lane >> 4;
    const int col0 = crank * COLS;
    const int A = p.A, T = p.T, K = p.K, B = p.B;

    extern __shared__ __align__(16) float smem[];
    float* W3s = smem;                         // [COLS][AP]
    float* W23s = W3s + COLS * AP;             // [COLS][AP]
    float* Wxs = W23s + COLS * AP;             // [AP][COLS]  W_in[a][col0 + j], rows a >= A zeroed
    float* actA = Wxs + AP * COLS;             // [R][LDA]    relu(u), all-gathered
    float* red = actA + R * LDA;               // [16][R][COLS] cross-warp partials (layer 0, then L1)
    float* cobs = red + R * H;                 // [R][COLS]   obs[r] @ W_in[A+td:, col0 + j]
    float* uown = cobs + R * COLS;             // [R][COLS]   raw u, own columns (residual)
    float* out1 = uown + R * COLS;             // [R][COLS]   relu(h1), own columns
    float* xs = out1 + R * COLS;               // [R][AP]     current x
    float* part = xs + R * AP;                 // [16][R][AP] partial eps of every CTA
    float* b1s = part + CS_C * R * AP;         // [COLS]
    float* b3s = b1s + COLS;                   // [AP]
    float* W1s = b3s + AP;                     // [16][KRW][COLS] resident k-rows of every warp's share of the W1 slice

    for (int chunk = cid; chunk < p.nchunks; chunk += nclusters) {
        const int row0 = chunk * R;
        // ---- initialise x (x_T injected or Philox slot 0)
#pragma unroll
        for (int q = 0; q < NE; ++q) {
            const int e = tid + q * CS_THREADS;
            if (e < R * AP) {
                const int r = e / AP, a = e % AP;
                float v = 0.f;
                if (a < A && row0 + r < B) {
                    v = p.xT ? p.xT[(size_t)(row0 + r) * A + a]
                             : philox_normal(p.seed, p.offset, p.row_offset + row0 + r, 0, a);
                    if (crank == 0 && p.chains && K == T) p.chains[((size_t)(row0 + r) * (K + 1)) * A + a] = v;
                }
                xs[e] = v;
            }
        }
        __syncthreads();
        int cur_net = -1;

        for (int i = 0; i < T; ++i) {
            const int t = T - 1 - i;
            const int net = (t < K && !p.use_base_policy) ? 1 : 0;
            const float* w = p.w[net];
            if (net != cur_net) {
                // ---- (re)load this net's resident slices and recompute its obs term
                for (int idx = tid; idx < CS_C * KRW * COLS; idx += CS_THREADS) {
                    const int wk = idx / (KRW * COLS), rem = idx % (KRW * COLS);
                    W1s[idx] = w[p.o.w1 + (size_t)(wk * KPW + rem / COLS) * H + col0 + rem % COLS];
                }
                for (int idx = tid; idx < COLS * AP; idx += CS_THREADS) {
                    int k = idx / AP, a = idx % AP;
                    W3s[idx] = a < A ? w[p.o.w3 + (size_t)(col0 + k) * A + a] : 0.f;
                    W23s[idx] = a < A ? p.w23[net][(size_t)(col0 + k) * A + a] : 0.f;
                }
                if (tid < COLS) b1s[tid] = w[p.o.b1 + col0 + tid];
                if (tid < AP) b3s[tid] = tid < A ? p.b23[net][tid] : 0.f;
                for (int idx = tid; idx < AP * COLS; idx += CS_THREADS) {
                    const int a = idx / COLS, j = idx % COLS;
                    Wxs[idx] = a < A ? w[p.o.win + (size_t)a * H + col0 + j] : 0.f;
                }
                if (tid < R * COLS) {
                    const int r = tid / COLS, j = tid % COLS;
                    float c = 0.f;
                    for (int jo = 0; jo < p.Do; ++jo) {
                        const float ov = (row0 + r < B) ? p.obs[(size_t)(row0 + r) * p.Do + jo] : 0.f;
                        c = fmaf(ov, w[p.o.win + (size_t)(A + p.td + jo) * H + col0 + j], c);
                    }
                    cobs[tid] = c;
                }
                cur_net = net;
                __syncthreads();
            }
            // the bias row of this step's own columns and this step's noise do not depend on the products: fetch them first
            const float btv = tid < R * COLS ? p.bt[net][(size_t)t * H + col0 + tid % COLS] : 0.f;
            float nz[NE];
#pragma unroll
            for (int q = 0; q < NE; ++q) {
                const int e = tid + q * CS_THREADS;
                nz[q] = 0.f;
                if (e < R * AP) {
                    const int r = e / AP, a = e % AP;
                    if (a < A && row0 + r < B) {
                        const int64_t row = row0 + r;
                        nz[q] = p.noise ? p.noise[((size_t)i * B + row) * A + a] : philox_normal(p.seed, p.offset, p.row_offset + row, 1 + i, a);
                    }
                }
            }
            // ---- L0, own columns: u[:, cols] = x @ W_in[0:AP, cols] (K split over the warps) + obs term + bt[t]
            {
                float acc[RH][NC];
#pragma unroll
                for (int rr = 0; rr < RH; ++rr)
#pragma unroll
                    for (int m = 0; m < NC; ++m) acc[rr][m] = 0.f;
#pragma unroll
                for (int kk = 0; kk < KW; ++kk) {
                    const int a = warp * KW + kk;
                    float wv[NC];
#pragma unroll
                    for (int m = 0; m < NC; ++m) wv[m] = Wxs[a * COLS + c16 + 16 * m];
#pragma unroll
                    for (int rr = 0; rr < RH; ++rr) {
                        const float xv = xs[(2 * rr + half) * AP + a];
#pragma unroll
                        for (int m = 0; m < NC; ++m) acc[rr][m] = fmaf(xv, wv[m], acc[rr][m]);
                    }
                }
#pragma unroll
                for (int rr = 0; rr < RH; ++rr)
#pragma unroll
                    for (int m = 0; m < NC; ++m) red[(warp * R + 2 * rr + half) * COLS + c16 + 16 * m] = acc[rr][m];
            }
            __syncthreads();
            if (tid < R * COLS) {
                const int r = tid / COLS, j = tid % COLS;
                float u = cobs[tid] + btv;
#pragma unroll
                for (int wr = 0; wr < 16; ++wr) u += red[(wr * R + r) * COLS + j];
                uown[tid] = u;
                const float v = fmaxf(u, 0.f);
#pragma unroll 1
                for (int dst = 0; dst < CS_C; ++dst) cluster.map_shared_rank(actA, dst)[r * LDA + col0 + j] = v;
            }
            cluster.sync();    // relu(u) of all H columns is in every CTA's actA
            // ---- L1 slice: h1[:, cols] = relu(u) @ W1[:, cols] + b1; this warp's k-rows warp * KPW .. + KPW, the first KRW resident
            {
                float acc[RH][NC];
#pragma unroll
                for (int rr = 0; rr < RH; ++rr)
#pragma unroll
                    for (int m = 0; m < NC; ++m) acc[rr][m] = 0.f;
                const float* ap = actA + half * LDA + warp * KPW;
                const float* Ws = W1s + warp * KRW * COLS + c16;
#pragma unroll 4
                for (int kk = 0; kk < KRW; kk += 4) {
                    float wv[4][NC];
#pragma unroll
                    for (int q = 0; q < 4; ++q)
#pragma unroll
                        for (int m = 0; m < NC; ++m) wv[q][m] = Ws[(kk + q) * COLS + 16 * m];
#pragma unroll
                    for (int rr = 0; rr < RH; ++rr) {
                        const float4 a = *reinterpret_cast<const float4*>(ap + 2 * rr * LDA + kk);
#pragma unroll
                        for (int m = 0; m < NC; ++m) {
                            acc[rr][m] = fmaf(a.x, wv[0][m], acc[rr][m]); acc[rr][m] = fmaf(a.y, wv[1][m], acc[rr][m]);
                            acc[rr][m] = fmaf(a.z, wv[2][m], acc[rr][m]); acc[rr][m] = fmaf(a.w, wv[3][m], acc[rr][m]);
                        }
                    }
                }
                const float* Wg = w + p.o.w1 + (size_t)(warp * KPW) * H + col0 + c16;
#pragma unroll 2
                for (int kk = KRW; kk < KPW; kk += 4) {
                    float wv[4][NC];
#pragma unroll
                    for (int q = 0; q < 4; ++q)
#pragma unroll
                        for (int m = 0; m < NC; ++m) wv[q][m] = __ldg(Wg + (size_t)(kk + q) * H + 16 * m);
#pragma unroll
                    for (int rr = 0; rr < RH; ++rr) {
                        const float4 a = *reinterpret_cast<const float4*>(ap + 2 * rr * LDA + kk);
#pragma unroll
                        for (int m = 0; m < NC; ++m) {
                            acc[rr][m] = fmaf(a.x, wv[0][m], acc[rr][m]); acc[rr][m] = fmaf(a.y, wv[1][m], acc[rr][m]);
                            acc[rr][m] = fmaf(a.z, wv[2][m], acc[rr][m]); acc[rr][m] = fmaf(a.w, wv[3][m], acc[rr][m]);
                        }
                    }
                }
#pragma unroll
                for (int rr = 0; rr < RH; ++rr)
#pragma unroll
                    for (int m = 0; m < NC; ++m) red[(warp * R + 2 * rr + half) * COLS + c16 + 16 * m] = acc[rr][m];
            }
            __syncthreads();
            if (tid < R * COLS) {
                const int r = tid / COLS, j = tid % COLS;
                float s = b1s[j];
#pragma unroll
                for (int wr = 0; wr < 16; ++wr) s += red[(wr * R + r) * COLS + j];
                out1[tid] = fmaxf(s, 0.f);
            }
            __syncthreads();
            // ---- partial output layer over this CTA's columns, written straight into the 16 CTAs' partial buffers
#pragma unroll
            for (int q = 0; q < NE; ++q) {
                const int e = tid + q * CS_THREADS;
                if (e < R * AP) {
                    const int r = e / AP, a = e % AP;
                    float s = 0.f;
#pragma unroll 16
                    for (int k = 0; k < COLS; ++k) s = fmaf(out1[r * COLS + k], W23s[k * AP + a], s);
                    float s2 = 0.f;
#pragma unroll 16
                    for (int k = 0; k < COLS; ++k) s2 = fmaf(uown[r * COLS + k], W3s[k * AP + a], s2);
                    s += s2;
#pragma unroll 1
                    for (int dst = 0; dst < CS_C; ++dst) cluster.map_shared_rank(part, dst)[crank * (R * AP) + e] = s;
                }
            }
            cluster.sync();
            // ---- posterior mean / clipped noise / x update (identical in all 16 CTAs)
#pragma unroll
            for (int q = 0; q < NE; ++q) {
                const int e = tid + q * CS_THREADS;
                if (e < R * AP) {
                    const int r = e / AP, a = e % AP;
                    if (a < A && row0 + r < B) {
                        float ev = b3s[a];
#pragma unroll
                        for (int src = 0; src < CS_C; ++src) ev += part[src * (R * AP) + e];
                        const int64_t row = row0 + r;
                        const float xn = ddpm_step_elem(xs[e], ev, nz[q], t, p.sch, T, p.hp, t == 0);
                        xs[e] = xn;
                        if (crank == 0) {
                            if (p.chains && t <= K) p.chains[((size_t)row * (K + 1) + (K - t)) * A + a] = xn;
                            if (t == 0) {
                                p.actions[(size_t)row * A + a] = xn;
                                if (p.raw_actions && a < p.act_cols)
                                    p.raw_actions[(size_t)row * p.act_cols + a] = env_unnormalize_action(xn, p.act_min[a % p.Da], p.act_max[a % p.Da]);
                            }
                        }
                    }
                }
            }
            __syncthreads();
        }
    }
    // no CTA may exit while peers can still write into its shared memory
    cluster.sync();
}
