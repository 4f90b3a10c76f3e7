// tcgen05 path (DPPO_PREC_BF16) for large row counts: host programs.  Forward / backward chains run on the fused
// layer-chain kernel (fused_chain.cuh) when the shapes allow it (ReLU at H = 256 / 512, Mish at H = 256, 64-wide h0),
// else every MLP layer is one tc::gemm_kernel launch; the weight gradients are one grouped tcgen05 launch on CTA pairs
// (tcp::dw_pair_kernel) or, in the deterministic mode, one split-K GEMM + fixed-order reduction per product.
//
// Data layout in HBM (all bf16 activations are row-major [rows][features]; nothing is transposed):
//   h0   [N][KP0]   = [ x (A) | obs (Do) | onehot(t) (T) | 1 | 0.. ]          KP0 = roundup(A+Do+T+1, 64)
//        The one-hot block turns the per-t layer-0 bias bt[t] (time-MLP output folded through W_in)
//        into T extra rows of the layer-0 weight, so the time embedding costs no epilogue work in
//        the forward pass and its gradient (per-t column sums of du) falls out of dW0 = h0^T du.
//        The ones column does the same for the critic's input-layer bias gradient.
//   a0,a1 [N][H]    post-activation outputs of layer 0 / block.l1 (operands of the next layer and of dW)
//   pre0,pre1       Mish only: pre-activation copies (per-layer path) / gates mish'(pre) (fused path);
//                   ReLU derivatives are bit masks m0, m1 [N][H/32] (fused path) or taken from a > 0
//   v    [N][H]     residual-block output  v = a1 W2 + b2 + u,  u = h0 W0 re-accumulated by K-concatenating
//                   [a1 | h0] against [W2 ; W0] instead of storing and re-reading u
//   eps  [N][A]     fp32 (feeds the fp32 loss kernels)
//   dv, dh1, du     [N][H] bf16 gradients; deps / dvalue are padded to [N][64] bf16
// Weights: fp32 masters stay in h->params; bf16 operand copies are rebuilt after every update:
//   w2w0 [(H+KP0)][H] = [W2 ; W0 rows in h0 order]   (MN-major B of the forward layers, K-major B of dX)
//   w1   [H][H],  w3t [64][H] = W3^T (zero padded),  w3p [H][128] = W3 (zero padded),  w1t / w2t = W1^T / W2^T
#pragma once
#include "common.cuh"
#include "simt_kernels.cuh"
#include "tc_gemm.cuh"
#include "fused_chain.cuh"
#include "tc_dw_pair.cuh"

typedef __nv_bfloat16 bf16;

struct TcNetW {
    bf16 *w2w0, *w1, *w3t, *w3p;
    bf16 *w1t, *w2t;       // W1^T, W2^T [out][in]: MN-major B operands of the fused backward chain (actors only)
    float* bias2;          // critic: b2 + b_in (the residual's input-layer bias rides with block.l2's)
    int H;
};
struct TcPpoPlan;
struct TcState {
    TcNetW net[4];
    int KP0;
    TcPpoPlan* plan;       // state of the begin / chunk / finish PPO step in flight (one per handle)
};

// ------------------------------------------------------------------ small kernels
// bt == nullptr: the T time rows of the layer-0 operand are written elsewhere (actor_prep_body's bt16 output)
__device__ __forceinline__ void tc_pack_actor_body(const size_t i0, const size_t stride, const float* __restrict__ w, ActorOff o, int A, int td, int Do, int T, int H, int KP0,
                                     const float* __restrict__ bt, bf16* __restrict__ w2w0, bf16* __restrict__ w1,
                                     bf16* __restrict__ w3t, bf16* __restrict__ w3p, bf16* __restrict__ w1t, bf16* __restrict__ w2t) {
    for (size_t i = i0; i < (size_t)H * H; i += stride) {
        w2w0[i] = __float2bfloat16(w[o.w2 + i]); w1[i] = __float2bfloat16(w[o.w1 + i]);
        const size_t r = i / H, c = i % H;            // transposed copies: coalesced writes, strided (L2-resident) reads
        w1t[i] = __float2bfloat16(w[o.w1 + c * H + r]); w2t[i] = __float2bfloat16(w[o.w2 + c * H + r]);
    }
    for (size_t i = i0; i < (size_t)KP0 * H; i += stride) {
        int k = (int)(i / H), c = (int)(i % H);
        float v = 0.f;
        if (k < A) v = w[o.win + (size_t)k * H + c];
        else if (k < A + Do) v = w[o.win + (size_t)(k + td) * H + c];
        else if (k < A + Do + T) { if (!bt) continue; v = bt[(size_t)(k - A - Do) * H + c]; }
        w2w0[(size_t)H * H + i] = __float2bfloat16(v);
    }
    for (size_t i = i0; i < (size_t)64 * H; i += stride) {
        int a = (int)(i / H), k = (int)(i % H);
        w3t[i] = __float2bfloat16(a < A ? w[o.w3 + (size_t)k * A + a] : 0.f);
    }
    for (size_t i = i0; i < (size_t)H * 128; i += stride) {
        int k = (int)(i / 128), a = (int)(i % 128);
        w3p[i] = __float2bfloat16(a < A ? w[o.w3 + (size_t)k * A + a] : 0.f);
    }
}
__global__ void tc_pack_actor_kernel(const float* __restrict__ w, ActorOff o, int A, int td, int Do, int T, int H, int KP0,
                                     const float* __restrict__ bt, bf16* __restrict__ w2w0, bf16* __restrict__ w1,
                                     bf16* __restrict__ w3t, bf16* __restrict__ w3p, bf16* __restrict__ w1t, bf16* __restrict__ w2t) {
    tc_pack_actor_body((size_t)blockIdx.x * blockDim.x + threadIdx.x, (size_t)gridDim.x * blockDim.x, w, o, A, td, Do, T, H, KP0, bt, w2w0, w1, w3t, w3p, w1t, w2t);
}
__device__ __forceinline__ void tc_pack_critic_body(const size_t i0, const size_t stride, const float* __restrict__ w, CriticOff o, int A, int Do, int Hc, int KP0,
                                      bf16* __restrict__ w2w0, bf16* __restrict__ w1, bf16* __restrict__ w3t,
                                      bf16* __restrict__ w3p, float* __restrict__ bias2, bf16* __restrict__ w1t, bf16* __restrict__ w2t) {
    for (size_t i = i0; i < (size_t)Hc * Hc; i += stride) {
        w2w0[i] = __float2bfloat16(w[o.w2 + i]); w1[i] = __float2bfloat16(w[o.w1 + i]);
        const size_t r = i / Hc, c = i % Hc;
        w1t[i] = __float2bfloat16(w[o.w1 + c * Hc + r]); w2t[i] = __float2bfloat16(w[o.w2 + c * Hc + r]);
    }
    for (size_t i = i0; i < (size_t)KP0 * Hc; i += stride) {
        int k = (int)(i / Hc), c = (int)(i % Hc);
        float v = (k >= A && k < A + Do) ? w[o.win + (size_t)(k - A) * Hc + c] : 0.f;
        w2w0[(size_t)Hc * Hc + i] = __float2bfloat16(v);
    }
    for (size_t i = i0; i < (size_t)64 * Hc; i += stride) { int a = (int)(i / Hc), k = (int)(i % Hc); w3t[i] = __float2bfloat16(a == 0 ? w[o.w3 + k] : 0.f); }
    for (size_t i = i0; i < (size_t)Hc * 128; i += stride) { int k = (int)(i / 128), a = (int)(i % 128); w3p[i] = __float2bfloat16(a == 0 ? w[o.w3 + k] : 0.f); }
    for (size_t i = i0; i < (size_t)Hc; i += stride) bias2[i] = w[o.b2 + i] + w[o.bin + i];
}
__global__ void tc_pack_critic_kernel(const float* __restrict__ w, CriticOff o, int A, int Do, int Hc, int KP0,
                                      bf16* __restrict__ w2w0, bf16* __restrict__ w1, bf16* __restrict__ w3t,
                                      bf16* __restrict__ w3p, float* __restrict__ bias2, bf16* __restrict__ w1t, bf16* __restrict__ w2t) {
    tc_pack_critic_body((size_t)blockIdx.x * blockDim.x + threadIdx.x, (size_t)gridDim.x * blockDim.x, w, o, A, Do, Hc, KP0, w2w0, w1, w3t, w3p, bias2, w1t, w2t);
}
// After the fine-tuning AdamW step: derived time tables of actor_ft, its bf16 operand copies and the critic's, in ONE launch
// (blocks [0,T): one denoising step's table row each | next na blocks: actor operands | rest: critic operands).
struct TcPrepPackArgs {
    const float* wa; ActorOff ao; const float* wc; CriticOff co; int A, td, Do, T, H, Hc, KP0, na, nc;
    float* sinemb; float* thpre; float* temb; float* bt;
    bf16 *a_w2w0, *a_w1, *a_w3t, *a_w3p, *a_w1t, *a_w2t;
    bf16 *c_w2w0, *c_w1, *c_w3t, *c_w3p, *c_w1t, *c_w2t; float* c_bias2;
};
__global__ void __launch_bounds__(256) tc_prep_pack_kernel(const TcPrepPackArgs a) {
    extern __shared__ float prep_sm[];
    const int b = blockIdx.x;
    if (b < a.T)
        actor_prep_body(b, prep_sm, WRead{a.wa}, a.ao, a.A, a.td, a.H, a.sinemb, a.thpre, a.temb, a.bt, a.a_w2w0 + (size_t)a.H * a.H + (size_t)(a.A + a.Do) * a.H);
    else if (b < a.T + a.na)
        tc_pack_actor_body((size_t)(b - a.T) * blockDim.x + threadIdx.x, (size_t)a.na * blockDim.x, a.wa, a.ao, a.A, a.td, a.Do, a.T, a.H, a.KP0, nullptr,
                           a.a_w2w0, a.a_w1, a.a_w3t, a.a_w3p, a.a_w1t, a.a_w2t);
    else
        tc_pack_critic_body((size_t)(b - a.T - a.na) * blockDim.x + threadIdx.x, (size_t)a.nc * blockDim.x, a.wc, a.co, a.A, a.Do, a.Hc, a.KP0,
                            a.c_w2w0, a.c_w1, a.c_w3t, a.c_w3p, a.c_bias2, a.c_w1t, a.c_w2t);
}
// Index-driven minibatch (train_ppo_diffusion_agent.py:292-312 without materialising it): row r of the minibatch is the
// (rollout row b, denoising index k) pair of flat[r] = b * K + k; the kernels below read the resident rollout buffers directly.
struct TcIdxView {
    const int* flat; int K; long long P;
    const float *chains, *obs, *olp, *ret, *val, *adv;      // [P][K+1][A], [P][Do], [P][K][A], [P], [P], [P]
    int* bad;                                                // set to 1 when an index lies outside [0, P*K)
};
// h0[r] = [x[r] | obs[r / obs_div] | onehot(t_r) | 1 | 0..]; one thread per 8 consecutive columns (16-byte store)
// chainK > 0: x is a chains tensor [B][chainK+1][A] and row r = b*chainK + k reads chains[b][k] (get_logprobs)
__global__ void tc_pack_h0_kernel(const float* __restrict__ x, const float* __restrict__ obs, const int* __restrict__ trow, int tconst,
                                  int N, int A, int Do, int T, int KP0, int obs_div, bf16* __restrict__ h0, int chainK = 0,
                                  const int* __restrict__ flat = nullptr, int flatK = 1, long long flatP = 0, int* __restrict__ bad = nullptr) {
    const int g8 = KP0 / 8;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * g8) return;
    const int r = (int)(i / g8), k0 = (int)(i % g8) * 8;
    // trow given: t = trow[r], or K-1-trow[r] when tconst = -K (denoising indices); else the constant tconst
    int t = trow ? (tconst < 0 ? -tconst - 1 - trow[r] : trow[r]) : tconst;
    size_t xrow = chainK > 0 ? (size_t)(r / chainK) * (chainK + 1) + (r % chainK) : (size_t)r;
    size_t orow = (size_t)(r / obs_div);
    if (flat) {   // index-driven: x = chains[b][k], obs = obs[b], t = K-1-k
        int f = flat[r];
        if (f < 0 || (long long)f >= flatP * flatK) { if (bad && k0 == 0) atomicOr(bad, 1); f = 0; }
        const int b = f / flatK, k = f % flatK;
        xrow = (size_t)b * (flatK + 1) + k; orow = (size_t)b; t = flatK - 1 - k;
    }
    __align__(16) bf16 o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int k = k0 + j;
        float v = 0.f;
        if (k < A) v = x ? x[xrow * A + k] : 0.f;
        else if (k < A + Do) v = obs[orow * Do + (k - A)];
        else if (k < A + Do + T) v = (k - A - Do == t) ? 1.f : 0.f;
        else if (k == A + Do + T) v = 1.f;
        o[j] = __float2bfloat16(v);
    }
    *reinterpret_cast<uint4*>(h0 + (size_t)r * KP0 + k0) = *reinterpret_cast<const uint4*>(o);
}
// dst[r][0:64] (bf16) = [src[r][0:ncols] | 0..]
__global__ void tc_pad64_kernel(const float* __restrict__ src, int N, int ncols, bf16* __restrict__ dst) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * 8) return;
    const int r = (int)(i >> 3), k0 = (int)(i & 7) * 8;
    __align__(16) bf16 o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = __float2bfloat16(k0 + j < ncols ? src[(size_t)r * ncols + k0 + j] : 0.f);
    *reinterpret_cast<uint4*>(dst + (size_t)r * 64 + k0) = *reinterpret_cast<const uint4*>(o);
}
// column sums of a bf16 matrix D[N][ncols] (ncols even, ncols/2 <= 256): part[blk][ncols]
__global__ void __launch_bounds__(256) tc_colsum_kernel(const bf16* __restrict__ D, int N, int ncols, int rows_per_block, float* __restrict__ part) {
    __shared__ float2 red[256];
    const int tpr = ncols / 2, groups = 256 / tpr;
    const int cg = threadIdx.x % tpr, rg = threadIdx.x / tpr;
    const int r0 = blockIdx.x * rows_per_block, r1 = min(N, r0 + rows_per_block);
    float2 acc = make_float2(0.f, 0.f);
    if (rg < groups) {
        for (int r = r0 + rg; r < r1; r += groups) {
            __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(D + (size_t)r * ncols + 2 * cg);
            float2 f = __bfloat1622float2(v);
            acc.x += f.x; acc.y += f.y;
        }
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x < tpr) {
        float2 s = red[threadIdx.x];
        for (int g = 1; g < groups; ++g) { float2 o = red[g * tpr + threadIdx.x]; s.x += o.x; s.y += o.y; }
        part[(size_t)blockIdx.x * ncols + 2 * threadIdx.x] = s.x;
        part[(size_t)blockIdx.x * ncols + 2 * threadIdx.x + 1] = s.y;
    }
}
// out[r][c] = sum_s part[s*stride + r*ld_in + c]   for r < rows, c < cols   (deterministic split-K reduction)
__global__ void tc_reduce2d_kernel(const float* __restrict__ part, int S, size_t stride, int rows, int cols, int ld_in,
                                   float* __restrict__ out, int ld_out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)rows * cols) return;
    const int r = (int)(i / cols), c = (int)(i % cols);
    float s = 0.f;
    for (int k = 0; k < S; ++k) s += part[(size_t)k * stride + (size_t)r * ld_in + c];
    out[(size_t)r * ld_out + c] = s;
}

// out[c] = sum_b part[b*stride + c]: one warp per column, lanes stride over the nb partial rows (deterministic)
// columns >= split (when out2 is given) go to out2[c - split]
__device__ __forceinline__ void tc_reduce_cols_body(const int bid, const float* __restrict__ part, int nb, size_t stride, int ncols,
                                                    float* __restrict__ out, int split, float* __restrict__ out2) {
    const int c = bid * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (c >= ncols) return;
    float s = 0.f;
    for (int b = lane; b < nb; b += 32) s += part[(size_t)b * stride + c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) { if (out2 && c >= split) out2[c - split] = s; else out[c] = s; }
}
// the same sums for MANY partial rows (the plane GEMM epilogues leave one row per 32 batch rows: 1563 at 50 000): a 512-thread block owns 32
// columns, lane = column, its 16 warps stride over the rows (every read a full 128-byte line), fixed-order combine through shared memory
__device__ __forceinline__ void tc_reduce_cols_wide_body(const int bid, const float* __restrict__ part, int nb, size_t stride, int ncols,
                                                         float* __restrict__ out, int split, float* __restrict__ out2) {
    __shared__ float red[16][33];
    const int lane = threadIdx.x & 31, rg = threadIdx.x >> 5, c = bid * 32 + lane;
    float sacc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) sacc[q] = 0.f;
    if (c < ncols) {
        int b = rg;
        for (; b + 112 < nb; b += 128) {          // eight independent loads in flight per thread
#pragma unroll
            for (int q = 0; q < 8; ++q) sacc[q] += part[(size_t)(b + 16 * q) * stride + c];
        }
        for (; b < nb; b += 16) sacc[0] += part[(size_t)b * stride + c];
    }
    red[rg][lane] = ((sacc[0] + sacc[1]) + (sacc[2] + sacc[3])) + ((sacc[4] + sacc[5]) + (sacc[6] + sacc[7]));
    __syncthreads();
    if (rg == 0 && c < ncols) {
        float s = 0.f;
#pragma unroll
        for (int g = 0; g < 16; ++g) s += red[g][lane];
        if (out2 && c >= split) out2[c - split] = s; else out[c] = s;
    }
}
__global__ void __launch_bounds__(256) tc_reduce_cols_kernel(const float* __restrict__ part, int nb, size_t stride, int ncols, float* __restrict__ out,
                                                             int split = 0, float* __restrict__ out2 = nullptr) {
    tc_reduce_cols_body(blockIdx.x, part, nb, stride, ncols, out, split, out2);
}

// Everything between the grouped weight-gradient GEMM and AdamW in ONE launch (tensor path, deferred mode): the eight small
// kernels are mutually independent, so block ranges take the roles - loss metrics | three column reductions (output-layer and
// hidden-layer bias gradients) | time-embedding backward | the two dW0 scatters | the critic's input-bias row.
struct TcTailArgs {
    int first[9];                                  // first block of role r; first[8] = grid size
    // metrics
    const double* bsum; int blocks_done; float inv_nglobal, frac_local; float* metrics;
    // column reductions (wide: the 32-columns-per-block body for many partial rows)
    int wide, wide3;
    const float* colb3; int ncol3; float* b3a; int split3; float* b3c;
    const float* cpa; int rows_a; int HA; float* b2a; float* b1a;
    const float* cpc; int rows_c; int HC; float* b2c; float* b1c;
    // time backward
    const float* w; ActorOff ao; int A, td, T, Do; const float* Gt; const float* sinemb; const float* thpre; const float* temb; float* dte; float* gr;
    // unpack
    const float* dw0a; float* gwin_a; const float* dw0c_obs; float* gwin_c; const float* dw0c_bias; float* gbin_c;
};
__global__ void __launch_bounds__(512) tc_ppo_tail_kernel(const TcTailArgs a) {
    pdl_grid_begin();
    extern __shared__ float tail_sm[];
    const int b = blockIdx.x;
    if (b < a.first[1]) ppo_metrics_body(a.bsum, a.blocks_done, a.inv_nglobal, a.frac_local, a.metrics);
    else if (b < a.first[2]) {
        if (a.wide3) tc_reduce_cols_wide_body(b - a.first[1], a.colb3, a.blocks_done, (size_t)a.ncol3, a.ncol3, a.b3a, a.split3, a.b3c);
        else tc_reduce_cols_body(b - a.first[1], a.colb3, a.blocks_done, (size_t)a.ncol3, a.ncol3, a.b3a, a.split3, a.b3c);
    }
    else if (b < a.first[3]) {
        if (a.wide) tc_reduce_cols_wide_body(b - a.first[2], a.cpa, a.rows_a, (size_t)2 * a.HA, 2 * a.HA, a.b2a, a.HA, a.b1a);
        else tc_reduce_cols_body(b - a.first[2], a.cpa, a.rows_a, (size_t)2 * a.HA, 2 * a.HA, a.b2a, a.HA, a.b1a);
    } else if (b < a.first[4]) {
        if (a.wide) tc_reduce_cols_wide_body(b - a.first[3], a.cpc, a.rows_c, (size_t)2 * a.HC, 2 * a.HC, a.b2c, a.HC, a.b1c);
        else tc_reduce_cols_body(b - a.first[3], a.cpc, a.rows_c, (size_t)2 * a.HC, 2 * a.HC, a.b2c, a.HC, a.b1c);
    }
    else if (b < a.first[5]) time_backward_body(b - a.first[4], tail_sm, a.w, a.ao, a.A, a.td, a.HA, a.T, a.Gt, a.sinemb, a.thpre, a.temb, a.dte, a.gr);
    else if (b < a.first[6]) unpack_dw0_body(b - a.first[5], a.dw0a, a.A, a.td, a.Do, a.HA, a.gwin_a);
    else if (b < a.first[7]) unpack_dw0_body(b - a.first[6], a.dw0c_obs, 0, 0, a.Do, a.HC, a.gwin_c);
    else { const int i = (b - a.first[7]) * blockDim.x + threadIdx.x; if (i < a.HC) a.gbin_c[i] = a.dw0c_bias[i]; }
}

// PPO loss + gradient seeds for the tensor path (diffusion_ppo.py:32-132), one thread per row, single pass:
// writes the padded bf16 seeds the backward chains consume (depsb / dvalb [N][64]), the metric partial sums, and the
// per-block column sums of deps / dvalue (output-layer bias gradients) - no fp32 deps round trip, no separate pad / colsum.
__global__ void __launch_bounds__(128) tc_ppo_loss_kernel(
    const float* __restrict__ prev, const float* __restrict__ nxt, const float* __restrict__ eps,
    const int* __restrict__ inds, const float* __restrict__ returns, const float* __restrict__ oldvalues,
    const float* __restrict__ advantages, const float* __restrict__ oldlogp, const float* __restrict__ newvalues,
    const float* __restrict__ advstats, const float* __restrict__ sch, PpoHyper hp, int N,
    bf16* __restrict__ depsb, bf16* __restrict__ dvalb, double* __restrict__ block_sums, float* __restrict__ col_part /*[blocks][A+1]*/) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    const int A = hp.A;
    double acc[5] = {0, 0, 0, 0, 0};
    float gout[32];
#pragma unroll
    for (int a = 0; a < 32; ++a) gout[a] = 0.f;
    float dv_out = 0.f;
    if (r < N) {
        const int ind = inds[r], t = hp.K - 1 - ind;
        const int nuse = min(hp.reward_horizon, A / hp.Da) * hp.Da;   // newlogprobs[:, :reward_horizon, :]
        const StepConst sc = step_const(sch, hp.T, t);
        const float sd = logprob_std(sc, hp.min_lp_std);
        const float lgs = 0.91893853320467274f + logf(sd);
        float newm = 0.f, oldm = 0.f;
        float zs[32]; uint32_t live = 0u;
#pragma unroll
        for (int a = 0; a < 32; ++a) {
            zs[a] = 0.f;
            if (a < nuse) {
                const size_t i = (size_t)r * A + a;
                float z; bool in;
                const float lp = logprob_elem_c(prev[i], eps[i], nxt[i], sc, sd, lgs, hp.dcv, &z, &in);
                newm += fminf(fmaxf(lp, hp.lp_lo), hp.lp_hi);
                oldm += fminf(fmaxf(oldlogp[i], hp.lp_lo), hp.lp_hi);
                zs[a] = z;
                if (lp >= hp.lp_lo && lp <= hp.lp_hi && in) live |= 1u << a;
            }
        }
        newm /= (float)nuse; oldm /= (float)nuse;
        const PpoRowPolicy p = ppo_row_policy(newm, oldm, advantages[r], advstats, ind, hp);
        const float gscale = p.dnew / (float)nuse / sd * sc.c1 * (-sc.srm1);
#pragma unroll
        for (int a = 0; a < 32; ++a) gout[a] = ((live >> a) & 1u) ? gscale * zs[a] : 0.f;
        const PpoRowValue vr = ppo_row_value(newvalues[r], returns[r], oldvalues + r, hp);
        dv_out = vr.seed;
        ppo_row_metrics(acc, p, vr.vl);
        // padded bf16 rows: [deps (A) | 0..] and [dvalue | 0..]
        uint4* drow = reinterpret_cast<uint4*>(depsb + (size_t)r * 64);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint4 u;
            u.x = fc::pack_bf16(gout[q * 8 + 0], gout[q * 8 + 1]); u.y = fc::pack_bf16(gout[q * 8 + 2], gout[q * 8 + 3]);
            u.z = fc::pack_bf16(gout[q * 8 + 4], gout[q * 8 + 5]); u.w = fc::pack_bf16(gout[q * 8 + 6], gout[q * 8 + 7]);
            drow[q] = u;
        }
#pragma unroll
        for (int q = 4; q < 8; ++q) drow[q] = make_uint4(0u, 0u, 0u, 0u);
        uint4* vrow = reinterpret_cast<uint4*>(dvalb + (size_t)r * 64);
        vrow[0] = make_uint4(fc::pack_bf16(dv_out, 0.f), 0u, 0u, 0u);
#pragma unroll
        for (int q = 1; q < 8; ++q) vrow[q] = make_uint4(0u, 0u, 0u, 0u);
    }
    // ---- block reductions: metric sums (double) and column sums of the seeds
    __shared__ double red[5][128];
    __shared__ float cred[4][33];
    for (int k = 0; k < 5; ++k) red[k][threadIdx.x] = acc[k];
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < 33; ++a) {
        float v = a < 32 ? gout[a < 32 ? a : 0] : dv_out;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if (lane == 0) cred[wrp][a] = v;
    }
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if (threadIdx.x < o) for (int k = 0; k < 5; ++k) red[k][threadIdx.x] += red[k][threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x < 5) block_sums[(size_t)blockIdx.x * 5 + threadIdx.x] = red[threadIdx.x][0];
    if (threadIdx.x <= A) {
        const int a = threadIdx.x < A ? threadIdx.x : 32;
        col_part[(size_t)blockIdx.x * (A + 1) + threadIdx.x] = cred[0][a] + cred[1][a] + cred[2][a] + cred[3][a];
    }
}

// The same loss with EIGHT lanes per row (A % 4 == 0, A <= 32): lane `sub` of a row owns elements [4 sub, 4 sub + 4) and reads them
// as one float4 per input array (coalesced; the thread-per-row kernel above walks 96-byte strides and leaves the SMs at ~10 warps).
// 32 rows per 256-thread block.  Row scalars are computed redundantly by the row's lanes after a 3-step shuffle reduction.
// LPR = 32 (split-precision mode, A % 4 == 0, 32 < A <= 128): a warp per row, 8 rows per block, seed rows 128 wide (the actor's NOP).
constexpr int LOSS8_ROWS = 32;
template <int LPR = 8>
__global__ void __launch_bounds__(256) tc_ppo_loss8_kernel(
    const float* __restrict__ prev, const float* __restrict__ nxt, const float* __restrict__ eps,
    const int* __restrict__ inds, const float* __restrict__ returns, const float* __restrict__ oldvalues,
    const float* __restrict__ advantages, const float* __restrict__ oldlogp, const float* __restrict__ newvalues,
    const float* __restrict__ advstats, const float* __restrict__ sch, PpoHyper hp, int N,
    bf16* __restrict__ depsb, bf16* __restrict__ dvalb, double* __restrict__ block_sums, float* __restrict__ col_part /*[blocks][A+1]*/,
    const TcIdxView iv, bf16* __restrict__ depsb_lo = nullptr, bf16* __restrict__ dvalb_lo = nullptr /* second planes (DPPO_PREC_BF16X3) */) {
    static_assert(LPR == 8 || LPR == 32, "eight lanes (A <= 32) or a warp (A <= 128) per row");
    constexpr int ROWS = 256 / LPR, DLD = LPR == 8 ? 64 : 128;     // rows per block; seed row width
    const int tid = threadIdx.x, sub = tid & (LPR - 1), lane = tid & 31, wrp = tid >> 5;
    const int r = blockIdx.x * ROWS + tid / LPR;
    const int A = hp.A, a0 = sub * 4;
    const bool row_ok = r < N;
    // where this row's inputs live: the materialised minibatch arrays, or (index-driven) the resident rollout buffers
    size_t prow = (size_t)r * A, nrow = prow, lrow = prow, srow = (size_t)r;
    int ind_r = 0;
    if (row_ok) {
        if (iv.flat) {
            int f = iv.flat[r];
            if (f < 0 || (long long)f >= iv.P * iv.K) f = 0;                 // flagged by the h0 pack kernel
            const size_t b = (size_t)(f / iv.K); ind_r = f % iv.K;
            prow = (b * (iv.K + 1) + ind_r) * A; nrow = prow + A; lrow = (b * iv.K + ind_r) * A; srow = b;
            prev = iv.chains; nxt = iv.chains; oldlogp = iv.olp; returns = iv.ret; oldvalues = iv.val; advantages = iv.adv;
        } else ind_r = inds[r];
    }
    const int nuse = min(hp.reward_horizon, A / hp.Da) * hp.Da;   // newlogprobs[:, :reward_horizon, :]
    float z[4] = {0.f, 0.f, 0.f, 0.f}, gq[4] = {0.f, 0.f, 0.f, 0.f};
    float newp = 0.f, oldp = 0.f, dv_out = 0.f, sd = 1.f;
    uint32_t live = 0u;
    double acc[5] = {0, 0, 0, 0, 0};
    int ind = 0;
    StepConst sc = {};
    if (row_ok) {
        ind = ind_r;
        sc = step_const(sch, hp.T, hp.K - 1 - ind);
        sd = logprob_std(sc, hp.min_lp_std);
        if (a0 < A) {
            const float lgs = 0.91893853320467274f + logf(sd);
            const float4 pv = *reinterpret_cast<const float4*>(prev + prow + a0), nx = *reinterpret_cast<const float4*>(nxt + nrow + a0);
            const float4 ep = *reinterpret_cast<const float4*>(eps + (size_t)r * A + a0), ol = *reinterpret_cast<const float4*>(oldlogp + lrow + a0);
            const float pvv[4] = {pv.x, pv.y, pv.z, pv.w}, nxv[4] = {nx.x, nx.y, nx.z, nx.w};
            const float epv[4] = {ep.x, ep.y, ep.z, ep.w}, olv[4] = {ol.x, ol.y, ol.z, ol.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                if (a0 + e < nuse) {
                    float zz; bool in;
                    const float lp = logprob_elem_c(pvv[e], epv[e], nxv[e], sc, sd, lgs, hp.dcv, &zz, &in);
                    newp += fminf(fmaxf(lp, hp.lp_lo), hp.lp_hi);
                    oldp += fminf(fmaxf(olv[e], hp.lp_lo), hp.lp_hi);
                    z[e] = zz;
                    if (lp >= hp.lp_lo && lp <= hp.lp_hi && in) live |= 1u << e;
                }
            }
        }
    }
#pragma unroll
    for (int off = 1; off < LPR; off <<= 1) { newp += __shfl_xor_sync(0xffffffffu, newp, off); oldp += __shfl_xor_sync(0xffffffffu, oldp, off); }
    if (row_ok) {
        const PpoRowPolicy p = ppo_row_policy(newp / (float)nuse, oldp / (float)nuse, advantages[srow], advstats, ind, hp);
        const float gscale = p.dnew / (float)nuse / sd * sc.c1 * (-sc.srm1);
#pragma unroll
        for (int e = 0; e < 4; ++e) gq[e] = ((live >> e) & 1u) ? gscale * z[e] : 0.f;
        // padded bf16 seed row [deps (A) | 0..]: this lane's 4 columns and 4 of the zero columns
        uint2* drow = reinterpret_cast<uint2*>(depsb + (size_t)r * DLD);
        drow[sub] = make_uint2(fc::pack_bf16(gq[0], gq[1]), fc::pack_bf16(gq[2], gq[3]));
        if (LPR == 8) drow[8 + sub] = make_uint2(0u, 0u);
        if (depsb_lo) {   // second plane: what the first one rounded away
            float lo[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) lo[e] = gq[e] - __bfloat162float(__float2bfloat16(gq[e]));
            uint2* lrow = reinterpret_cast<uint2*>(depsb_lo + (size_t)r * DLD);
            lrow[sub] = make_uint2(fc::pack_bf16(lo[0], lo[1]), fc::pack_bf16(lo[2], lo[3]));
            if (LPR == 8) lrow[8 + sub] = make_uint2(0u, 0u);
        }
        if (sub == 0) {
            const PpoRowValue vr = ppo_row_value(newvalues[r], returns[srow], oldvalues + srow, hp);
            dv_out = vr.seed;
            ppo_row_metrics(acc, p, vr.vl);
        }
        // padded bf16 seed row [dvalue | 0..]: 16 bytes per lane
        uint4* vrow = reinterpret_cast<uint4*>(dvalb + (size_t)r * 64);
        if (sub < 8) vrow[sub] = sub == 0 ? make_uint4(fc::pack_bf16(dv_out, 0.f), 0u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
        if (dvalb_lo && sub < 8) {
            uint4* lrow = reinterpret_cast<uint4*>(dvalb_lo + (size_t)r * 64);       // dv_out lives in the row's lane 0
            lrow[sub] = sub == 0 ? make_uint4(fc::pack_bf16(dv_out - __bfloat162float(__float2bfloat16(dv_out)), 0.f), 0u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
        }
    }
    // ---- block reductions: rows of a warp (lanes differing in bits 3,4), then the 8 warps through shared memory
    __shared__ double red[5][8];
    __shared__ float cred[8][4 * LPR + 1];
#pragma unroll
    for (int off = LPR; off < 32; off <<= 1) {
#pragma unroll
        for (int k = 0; k < 5; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], off);
#pragma unroll
        for (int e = 0; e < 4; ++e) gq[e] += __shfl_xor_sync(0xffffffffu, gq[e], off);
        dv_out += __shfl_xor_sync(0xffffffffu, dv_out, off);
    }
    if (lane == 0) { for (int k = 0; k < 5; ++k) red[k][wrp] = acc[k]; cred[wrp][4 * LPR] = dv_out; }
    if (lane < LPR) { for (int e = 0; e < 4; ++e) cred[wrp][lane * 4 + e] = gq[e]; }
    __syncthreads();
    if (tid < 5) { double t = 0; for (int w = 0; w < 8; ++w) t += red[tid][w]; block_sums[(size_t)blockIdx.x * 5 + tid] = t; }
    if (tid <= A) {
        const int a = tid < A ? tid : 4 * LPR;
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += cred[w][a];
        col_part[(size_t)blockIdx.x * (A + 1) + tid] = t;
    }
}

// ------------------------------------------------------------------ state
static int tc_init(dppo_handle* h) {
    const Geom& g = h->g;
    TcState* st = new TcState();
    memset(st, 0, sizeof(*st));
    h->tc = st;
    st->KP0 = round_up(g.A + g.Do + g.T + 1, 64);
    if ((g.H % 64) || (g.Hc % 64) || g.A > 32) return 0;    // shapes the tensor path does not cover: stays on FFMA
    for (int net = 0; net < 4; ++net) {
        TcNetW& w = st->net[net];
        const int H = net == DPPO_NET_CRITIC ? g.Hc : g.H;
        w.H = H;
        CUDA_TRY(cudaMalloc(&w.w2w0, (size_t)(H + st->KP0) * H * sizeof(bf16)));
        CUDA_TRY(cudaMalloc(&w.w1, (size_t)H * H * sizeof(bf16)));
        CUDA_TRY(cudaMalloc(&w.w3t, (size_t)64 * H * sizeof(bf16)));
        CUDA_TRY(cudaMalloc(&w.w1t, (size_t)H * H * sizeof(bf16)));
        CUDA_TRY(cudaMalloc(&w.w2t, (size_t)H * H * sizeof(bf16)));
        CUDA_TRY(cudaMalloc(&w.w3p, (size_t)H * 128 * sizeof(bf16)));
        CUDA_TRY(cudaMalloc(&w.bias2, (size_t)H * sizeof(float)));
    }
    return 0;
}
static void tc_destroy(dppo_handle* h) {
    if (!h->tc) return;
    for (int net = 0; net < 4; ++net) {
        TcNetW& w = h->tc->net[net];
        cudaFree(w.w2w0); cudaFree(w.w1); cudaFree(w.w3t); cudaFree(w.w3p); cudaFree(w.bias2); cudaFree(w.w1t); cudaFree(w.w2t);
    }
    delete h->tc; h->tc = nullptr;
}
static bool tc_shapes_ok(const dppo_handle* h) { return h->tc && h->tc->net[0].w1 != nullptr; }
static const int TC_MIN_ROWS = 2048;
static bool tc_eligible(const dppo_handle* h, int rows) {
    return h->cfg.precision == DPPO_PREC_BF16 && tc_shapes_ok(h) && rows >= TC_MIN_ROWS;
}
// rebuild the bf16 operand copies of one net (after set_weights / an optimizer step)
static int tc_refresh_net(dppo_handle* h, int net, cudaStream_t s) {
    if (h->cfg.precision != DPPO_PREC_BF16 || !tc_shapes_ok(h)) return 0;
    const Geom& g = h->g; TcNetW& w = h->tc->net[net];
    if (net == DPPO_NET_CRITIC)
        tc_pack_critic_kernel<<<128, 256, 0, s>>>(h->net_w[net], g.co, g.A, g.Do, g.Hc, h->tc->KP0, w.w2w0, w.w1, w.w3t, w.w3p, w.bias2, w.w1t, w.w2t);
    else
        tc_pack_actor_kernel<<<256, 256, 0, s>>>(h->net_w[net], g.ao, g.A, g.td, g.Do, g.T, g.H, h->tc->KP0, h->ad[net].bt, w.w2w0, w.w1, w.w3t, w.w3p, w.w1t, w.w2t);
    h->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) DPPO_FAIL(-3, "tc pack launch failed: %s", cudaGetErrorString(e));
    return 0;
}

// prep_net(ACTOR_FT) + prep_net(CRITIC) of the PPO update in one launch (tensor mode)
static int tc_prep_pack_ft_critic(dppo_handle* h, cudaStream_t s) {
    const Geom& g = h->g; TcNetW& wa = h->tc->net[DPPO_NET_ACTOR_FT]; TcNetW& wc = h->tc->net[DPPO_NET_CRITIC];
    const ActorDerived& d = h->ad[DPPO_NET_ACTOR_FT];
    TcPrepPackArgs a;
    a.wa = h->net_w[DPPO_NET_ACTOR_FT]; a.ao = g.ao; a.wc = h->net_w[DPPO_NET_CRITIC]; a.co = g.co;
    a.A = g.A; a.td = g.td; a.Do = g.Do; a.T = g.T; a.H = g.H; a.Hc = g.Hc; a.KP0 = h->tc->KP0; a.na = 256; a.nc = 128;
    a.sinemb = d.sinemb; a.thpre = d.thpre; a.temb = d.temb; a.bt = d.bt;
    a.a_w2w0 = wa.w2w0; a.a_w1 = wa.w1; a.a_w3t = wa.w3t; a.a_w3p = wa.w3p; a.a_w1t = wa.w1t; a.a_w2t = wa.w2t;
    a.c_w2w0 = wc.w2w0; a.c_w1 = wc.w1; a.c_w3t = wc.w3t; a.c_w3p = wc.w3p; a.c_w1t = wc.w1t; a.c_w2t = wc.w2t; a.c_bias2 = wc.bias2;
    h->w0p_dirty[DPPO_NET_ACTOR_FT] = 1; h->w0p_dirty[DPPO_NET_CRITIC] = 1;
    tc_prep_pack_kernel<<<g.T + a.na + a.nc, 256, 4 * g.td * sizeof(float), s>>>(a);
    h->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) DPPO_FAIL(-3, "tc prep/pack launch failed: %s", cudaGetErrorString(e));
    return 0;
}

#define TC_KCHECK(h) do { (h)->launches++; cudaError_t _e = cudaGetLastError(); if (_e != cudaSuccess) { \
    dppo_set_error("kernel launch failed at %s:%d: %s", __FILE__, __LINE__, cudaGetErrorString(_e)); return -3; } } while (0)
static inline int tc_nblk(size_t n, int b) { return (int)((n + b - 1) / b); }

// ------------------------------------------------------------------ fused layer-chain programs (fused_chain.cuh)
// one residual MLP as the fused kernel sees it
struct FcNet { int net, H, act1 /*1 ReLU, 2 Mish*/, NO, din /*un-padded input width*/; const float *b0, *b1, *b2, *b3; };
static FcNet fc_actor_net(const dppo_handle* h, int net) {
    const Geom& g = h->g; const float* w = h->net_w[net];
    FcNet n; n.net = net; n.H = g.H; n.act1 = h->cfg.actor_act + 1; n.NO = g.A; n.din = g.Din;
    n.b0 = nullptr; n.b1 = w + g.ao.b1; n.b2 = w + g.ao.b2; n.b3 = w + g.ao.b3;    // b_in rides in W0's one-hot rows (bt table)
    return n;
}
static FcNet fc_critic_net(const dppo_handle* h) {
    const Geom& g = h->g; const float* w = h->net_w[DPPO_NET_CRITIC];
    FcNet n; n.net = DPPO_NET_CRITIC; n.H = g.Hc; n.act1 = h->cfg.critic_act + 1; n.NO = 1; n.din = g.Do;
    n.b0 = w + g.co.bin; n.b1 = w + g.co.b1; n.b2 = h->tc->net[DPPO_NET_CRITIC].bias2; n.b3 = w + g.co.b3;
    return n;
}
// shapes the fused kernel covers: ReLU at H = 256 / 512, Mish at H = 256 (the gate buffer needs the shared memory)
static bool fc_net_ok(const dppo_handle* h, const FcNet& n) {
    if (!tc_shapes_ok(h) || h->tc->KP0 != 64 || h->force_path == 3 || n.NO > 32) return false;
    if (n.act1 == 1) return n.H == 512 || n.H == 256;
    if (n.act1 == 2) return n.H == 256;
    return false;
}
static bool fc_ok(const dppo_handle* h) { return fc_net_ok(h, fc_actor_net(h, DPPO_NET_ACTOR)); }
static bool fc_critic_ok(const dppo_handle* h) { return fc_net_ok(h, fc_critic_net(h)); }

static int fc_weight_maps(const dppo_handle* h, const FcNet& n, CUtensorMap* m) {
    const TcNetW& W = h->tc->net[n.net]; const int H = n.H;
    DPPO_TRY(fc::weight_map(&m[0], W.w2w0, H + 64, H, H));
    DPPO_TRY(fc::weight_map(&m[1], W.w1, H, H, H));
    DPPO_TRY(fc::weight_map(&m[2], W.w3p, H, 128, 128));      // a CTA pair splits N: the output layer is padded to 128 columns
    return 0;
}
// forward program: L0 act(H0 W0 + b0), L1 act(X W1 + b1), L2 X W2 + H0 W0 + b2, L3 X W3 + b3; weight maps at m[wbase..wbase+2]
static void fc_fwd_layers(const dppo_handle* h, const FcNet& n, int wbase, fc::Layer* L) {
    const int H = n.H;
    memset(L, 0, sizeof(fc::Layer) * fc::MAXL);
    for (int i = 0; i < fc::MAXL; ++i) { L[i].store_map = -1; L[i].gate_store_map = -1; L[i].gate_load_map = -1; L[i].colsum_slot = -1; }
    L[0].a_src = 0; L[0].wmap = wbase; L[0].wrow_h0 = H; L[0].n = H; L[0].bias = n.b0; L[0].act = n.act1;
    L[1].a_src = 1; L[1].wmap = wbase + 1; L[1].n = H; L[1].bias = n.b1; L[1].act = n.act1;
    L[2].a_src = 2; L[2].wmap = wbase; L[2].wrow_h0 = H; L[2].n = H; L[2].bias = n.b2; L[2].h0_last = 1;
    L[3].a_src = 1; L[3].wmap = wbase + 2; L[3].n = 128; L[3].bias = n.b3;
}
// algorithmic flops (SURVEY.md 8d: un-padded dims, time-MLP excluded): forward F = 2 (din H + 2 H^2 + H NO) per row
static double fc_fwd_flops(const FcNet& n, double rows) { const double H = n.H; return 2.0 * rows * (n.din * H + 2.0 * H * H + H * n.NO); }
static void fc_common(dppo_handle* h, fc::Params& p, int N, int NO) {
    const Geom& g = h->g;
    memset(&p, 0, sizeof(p));
    p.rows = N; p.A = NO; p.Do = g.Do; p.T = g.T; p.K = g.K; p.sch = h->sched;
    p.dcv = h->cfg.denoised_clip_value; p.min_lp_std = h->cfg.min_logprob_denoising_std;
    // dev tool: each chain launch gets its own slot of [sm_count][8] counters (16 slots, round robin)
    p.dbg = h->chain_dbg ? h->chain_dbg + (size_t)(h->chain_dbg_idx++ & 15) * h->sm_count * 8 : nullptr;
}
// inference forward from a packed h0: final = output store (eps / value) or Gaussian log-prob
static int fc_infer(dppo_handle* h, cudaStream_t s, const FcNet& n, const bf16* h0, int N, int mode, float* out,
                    const float* prev, const float* next, const float* chains, const int* trow) {
    fc::Maps maps; fc::Params p; fc_common(h, p, N, n.NO);
    DPPO_TRY(fc::rowtile_map(&maps.m[0], h0, N, 64));
    DPPO_TRY(fc_weight_maps(h, n, &maps.m[1]));
    for (int i = 4; i < fc::NMAPS; ++i) maps.m[i] = maps.m[0];
    p.nlayers = 4; p.final_mode = mode; p.h0_from_tma = 1;
    fc_fwd_layers(h, n, 1, p.L[0]);
    p.out = out; p.prev = prev; p.next = next; p.chains = chains; p.trow = trow;
    return fc::launch_chain(h, s, n.H, maps, p, fc_fwd_flops(n, N));
}
static int fc_actor_infer(dppo_handle* h, cudaStream_t s, int net, const bf16* h0, int N, int mode, float* out,
                          const float* prev, const float* next, const float* chains, const int* trow) {
    return fc_infer(h, s, fc_actor_net(h, net), h0, N, mode, out, prev, next, chains, trow);
}
// training forward: output + the tensors the backward needs in HBM via TMA store: a0, a1, v and either the ReLU bit
// masks (m0, m1) or the Mish gates mish'(pre-activation) (g0, g1)
static int fc_train_fwd(dppo_handle* h, cudaStream_t s, const FcNet& n, const bf16* h0, int N, bf16* a0, bf16* a1, bf16* v,
                        uint32_t* m0, uint32_t* m1, bf16* g0, bf16* g1, float* out) {
    const int H = n.H;
    fc::Maps maps; fc::Params p; fc_common(h, p, N, n.NO);
    DPPO_TRY(fc::rowtile_map(&maps.m[0], h0, N, 64));
    DPPO_TRY(fc_weight_maps(h, n, &maps.m[1]));
    DPPO_TRY(fc::rowtile_map(&maps.m[4], a0, N, H));
    DPPO_TRY(fc::rowtile_map(&maps.m[5], a1, N, H));
    DPPO_TRY(fc::rowtile_map(&maps.m[6], v, N, H));
    maps.m[7] = maps.m[0]; maps.m[8] = maps.m[0]; maps.m[9] = maps.m[0];
    p.nlayers = 4; p.final_mode = fc::FINAL_EPS; p.h0_from_tma = 1;
    fc_fwd_layers(h, n, 1, p.L[0]);
    p.L[0][0].store_map = 4; p.L[0][1].store_map = 5; p.L[0][2].store_map = 6;
    if (n.act1 == 1) { p.L[0][0].mask_out = m0; p.L[0][1].mask_out = m1; }
    else {
        DPPO_TRY(fc::rowtile_map(&maps.m[7], g0, N, H));
        DPPO_TRY(fc::rowtile_map(&maps.m[8], g1, N, H));
        p.L[0][0].gate_store_map = 7; p.L[0][1].gate_store_map = 8;
    }
    p.out = out;
    return fc::launch_chain(h, s, H, maps, p, fc_fwd_flops(n, N));
}
// backward chain: dv = dout W3^T, dh1 = (dv W2^T) . act'(h1), du = (dh1 W1^T) . act'(u)
// (du excludes the residual path: dW0 adds h0^T dv)
// colsum_part [sm_count][2][H]: per-CTA column sums of dv (slot 0 = db2) and dh1 (slot 1 = db1), reduced by the caller
static int fc_bwd(dppo_handle* h, cudaStream_t s, const FcNet& n, const bf16* doutb, int N, const uint32_t* m0, const uint32_t* m1,
                  const bf16* g0, const bf16* g1, bf16* dv, bf16* dh1, bf16* du, float* colsum_part) {
    const int H = n.H; const TcNetW& W = h->tc->net[n.net];
    fc::Maps maps; fc::Params p; fc_common(h, p, N, n.NO);
    DPPO_TRY(fc::rowtile_map(&maps.m[0], doutb, N, 64));
    DPPO_TRY(fc::weight_map(&maps.m[1], W.w3t, 64, H, H));
    DPPO_TRY(fc::weight_map(&maps.m[2], W.w2t, H, H, H));
    DPPO_TRY(fc::weight_map(&maps.m[3], W.w1t, H, H, H));
    DPPO_TRY(fc::rowtile_map(&maps.m[4], dv, N, H));
    DPPO_TRY(fc::rowtile_map(&maps.m[5], dh1, N, H));
    DPPO_TRY(fc::rowtile_map(&maps.m[6], du, N, H));
    maps.m[7] = maps.m[0]; maps.m[8] = maps.m[0]; maps.m[9] = maps.m[0];
    p.nlayers = 3; p.final_mode = fc::FINAL_STORE; p.h0_from_tma = 1;
    fc::Layer* L = p.L[0];
    memset(L, 0, sizeof(fc::Layer) * fc::MAXL);
    for (int i = 0; i < fc::MAXL; ++i) { L[i].store_map = -1; L[i].gate_store_map = -1; L[i].gate_load_map = -1; L[i].colsum_slot = -1; }
    L[0].a_src = 0; L[0].wmap = 1; L[0].wrow_h0 = 0; L[0].n = H; L[0].h0_last = 1; L[0].store_map = 4; L[0].colsum_slot = 0;
    L[1].a_src = 1; L[1].wmap = 2; L[1].n = H; L[1].store_map = 5; L[1].colsum_slot = 1;
    p.colsum_part = colsum_part;
    L[2].a_src = 1; L[2].wmap = 3; L[2].n = H; L[2].store_map = 6;
    if (n.act1 == 1) { L[1].mask_in = m1; L[2].mask_in = m0; }
    else {
        DPPO_TRY(fc::rowtile_map(&maps.m[7], g1, N, H));
        DPPO_TRY(fc::rowtile_map(&maps.m[8], g0, N, H));
        L[1].gate_load_map = 7; L[2].gate_load_map = 8;
    }
    return fc::launch_chain(h, s, H, maps, p, 2.0 * N * ((double)n.NO * H + 2.0 * H * H));
}
// VPGDiffusion.call for large batches: the whole T-step chain in ONE launch
static int fc_sample(dppo_handle* h, cudaStream_t s, const float* obs, int B, int use_base, SampleHyper hp, uint64_t seed,
                     uint64_t offset, int64_t row_offset, const float* xT, const float* noise, float* actions, float* chains) {
    const FcNet nb = fc_actor_net(h, DPPO_NET_ACTOR), nf = fc_actor_net(h, DPPO_NET_ACTOR_FT);
    fc::Maps maps; fc::Params p; fc_common(h, p, B, nb.NO);
    DPPO_TRY(fc_weight_maps(h, nb, &maps.m[1]));
    DPPO_TRY(fc_weight_maps(h, nf, &maps.m[4]));
    maps.m[0] = maps.m[1]; maps.m[7] = maps.m[1]; maps.m[8] = maps.m[1]; maps.m[9] = maps.m[1];
    p.nlayers = 4; p.final_mode = fc::FINAL_SAMPLE; p.h0_from_tma = 0;
    fc_fwd_layers(h, nb, 1, p.L[0]);
    fc_fwd_layers(h, nf, 4, p.L[1]);
    p.obs = obs; p.xT = xT; p.noise = noise; p.actions = actions; p.chains_out = chains; p.hp = hp; p.use_base_policy = use_base;
    p.seed = seed; p.offset = offset; p.row_offset = row_offset;
    return fc::launch_chain(h, s, nb.H, maps, p, fc_fwd_flops(nb, B) * h->g.T);
}

// ------------------------------------------------------------------ GEMM helpers
static tc::Operand opK(const bf16* p, int64_t mn, int64_t k, int64_t ld) { return tc::Operand{p, false, mn, k, ld}; }
static tc::Operand opMN(const bf16* p, int64_t mn, int64_t k, int64_t ld) { return tc::Operand{p, true, mn, k, ld}; }
static tc::Gemm gemm_of(tc::Operand A, tc::Operand B, int M, int N) {
    tc::Gemm g; memset(&g, 0, sizeof(g));
    g.A = A; g.B = B; g.M = M; g.N = N; g.splits = 1; g.epi.M = M; g.epi.N = N;
    return g;
}
static int tc_run(dppo_handle* h, cudaStream_t s, const tc::Gemm& g) { int r = tc::launch(h, s, g); return r < 0 ? r : 0; }

// one residual MLP (actor: ReLU, NO = A; critic: Mish, NO = 1) on N rows
struct TcMlp {
    const TcNetW* W; int H, NO, act1, KP0;
    const float *b0, *b1, *b2, *b3;       // fp32 biases (b0 null for the actor: bt rides in W0's one-hot rows)
    const bf16* h0;
    bf16 *a0, *a1, *v, *pre0, *pre1;      // pre* only when act1 == 2
    float* out;                            // [N][NO] fp32
    bf16 *dv, *dh1, *du;                   // backward
    uint32_t *m0, *m1;                     // fused chain: ReLU bit masks [N][H/32] of layer 0 / block.l1
    int fused, net, din;                   // fused: runs on the fused layer-chain kernel; din: un-padded input width
    float* cpart;                          // fused backward: where the per-CTA bias column sums go ([sm][2][H]); null = reduce at once
};
// the same MLP program on rows [r0, ...) of its per-row buffers
static TcMlp tc_mlp_at(const TcMlp& m, size_t r0) {
    TcMlp o = m;
    const size_t e = r0 * (size_t)m.H;
    if (o.h0) o.h0 += r0 * (size_t)m.KP0;
    if (o.a0) o.a0 += e; if (o.a1) o.a1 += e; if (o.v) o.v += e; if (o.pre0) o.pre0 += e; if (o.pre1) o.pre1 += e;
    if (o.dv) o.dv += e; if (o.dh1) o.dh1 += e; if (o.du) o.du += e;
    if (o.out) o.out += r0 * (size_t)m.NO;
    if (o.m0) o.m0 += r0 * (size_t)(m.H / 32); if (o.m1) o.m1 += r0 * (size_t)(m.H / 32);
    return o;
}
static void tc_mlp_take(dppo_handle* h, int N, TcMlp& m, bool bwd) {
    const size_t n = (size_t)N * m.H;
    m.a0 = ws_take<bf16>(h, n); m.a1 = ws_take<bf16>(h, n); m.v = ws_take<bf16>(h, n);
    m.pre0 = m.pre1 = nullptr;
    if (m.act1 == 2) { m.pre0 = ws_take<bf16>(h, n); m.pre1 = ws_take<bf16>(h, n); }
    m.dv = m.dh1 = m.du = nullptr;
    if (bwd) { m.dv = ws_take<bf16>(h, n); m.dh1 = ws_take<bf16>(h, n); m.du = ws_take<bf16>(h, n); }
    m.m0 = ws_take<uint32_t>(h, (size_t)N * (m.H / 32)); m.m1 = ws_take<uint32_t>(h, (size_t)N * (m.H / 32));
}
static int tc_mlp_forward(dppo_handle* h, cudaStream_t s, const TcMlp& m, int N) {
    const int H = m.H, KP0 = m.KP0; const TcNetW& W = *m.W;
    if (m.fused) return fc_train_fwd(h, s, m.net == DPPO_NET_CRITIC ? fc_critic_net(h) : fc_actor_net(h, m.net), m.h0, N, m.a0, m.a1, m.v,
                                     m.m0, m.m1, m.pre0, m.pre1, m.out);     // pre0 / pre1 hold the Mish gates on this path
    // L0: a0 = act(h0 W0 (+ b0))
    tc::Gemm g = gemm_of(opK(m.h0, N, KP0, KP0), opMN(W.w2w0 + (size_t)H * H, H, KP0, H), N, H);
    g.epi.bias = m.b0; g.epi.act = m.act1; g.epi.out_bf16 = m.a0; g.epi.ld_bf16 = H; g.epi.out_pre = m.pre0; g.epi.ld_pre = H;
    DPPO_TRY(tc_run(h, s, g));
    // L1: a1 = act(a0 W1 + b1)
    g = gemm_of(opK(m.a0, N, H, H), opMN(W.w1, H, H, H), N, H);
    g.epi.bias = m.b1; g.epi.act = m.act1; g.epi.out_bf16 = m.a1; g.epi.ld_bf16 = H; g.epi.out_pre = m.pre1; g.epi.ld_pre = H;
    DPPO_TRY(tc_run(h, s, g));
    // L2 + residual: v = [a1 | h0] [W2 ; W0] + b2 (+ b0)
    g = gemm_of(opK(m.a1, N, H, H), opMN(W.w2w0, H, H + KP0, H), N, H);
    g.A2 = opK(m.h0, N, KP0, KP0);
    g.epi.bias = m.b2; g.epi.out_bf16 = m.v; g.epi.ld_bf16 = H;
    DPPO_TRY(tc_run(h, s, g));
    // L3: out = v W3 + b3
    g = gemm_of(opK(m.v, N, H, H), opK(W.w3t, 32, H, H), N, m.NO);
    g.epi.bias = m.b3; g.epi.out_f32 = m.out; g.epi.ld_f32 = m.NO;
    DPPO_TRY(tc_run(h, s, g));
    return 0;
}
static int tc_splits_for(const dppo_handle* h, int M, int N, int rows) {
    const int BN = N > 128 ? 256 : (N > 64 ? 128 : 64);
    const int tiles = ((M + 127) / 128) * ((N + BN - 1) / BN);
    int splits = h->sm_count / tiles; if (splits < 1) splits = 1;
    const int kb = (rows + 63) / 64;
    int maxs = kb / 4; if (maxs < 1) maxs = 1;          // at least 4 k-blocks of work per split
    if (splits > maxs) splits = maxs;
    if (splits > 64) splits = 64;
    return splits;
}
// dW[M][ncols] (+)= X^T D  (X [rows][M] bf16, D [rows][Nd] bf16), split-K over the rows (+ X^T D2 when D2 is given).
// Default: every split CTA accumulates its tile into `out` with red.global.add.f32 (out must be zeroed beforehand; the
// summation order, hence the last bits, vary run to run).  DPPO_DETERMINISTIC=1: partial tiles + a fixed-order reduction.
static int tc_dw(dppo_handle* h, cudaStream_t s, const bf16* X, int M, const bf16* D, int Nd, int rows, float* part,
                 float* out, int out_rows, int out_cols, int ld_out, const bf16* D2 = nullptr, int alg_rows_in = -1) {
    const int alg_rows = alg_rows_in >= 0 ? alg_rows_in : out_rows;
    tc::Gemm g = gemm_of(opMN(X, M, rows, M), opMN(D, Nd, rows, Nd), M, Nd);
    g.splits = tc_splits_for(h, M, Nd, rows);
    g.alg_flops = 2.0 * (double)rows * (double)alg_rows * (double)out_cols;
    if (!h->deterministic) {
        g.epi.M = out_rows; g.epi.N = out_cols;
        g.epi.out_f32 = out; g.epi.ld_f32 = ld_out; g.epi.f32_atomic = 1;
        int S = tc::launch(h, s, g);
        if (S < 0) return S;
        if (D2) { g.B = opMN(D2, Nd, rows, Nd); g.alg_flops = 1.0; S = tc::launch(h, s, g); if (S < 0) return S; }   // residual path: not algorithmic work
        return 0;
    }
    g.epi.out_f32 = part; g.epi.ld_f32 = Nd; g.epi.split_stride = (size_t)M * Nd;
    int S = tc::launch(h, s, g);
    if (S < 0) return S;
    if (D2) {
        g.B = opMN(D2, Nd, rows, Nd);
        g.epi.out_f32 = part + (size_t)S * M * Nd;
        int S2 = tc::launch(h, s, g);
        if (S2 < 0) return S2;
        S += S2;
    }
    tc_reduce2d_kernel<<<tc_nblk((size_t)out_rows * out_cols, 256), 256, 0, s>>>(part, S, (size_t)M * Nd, out_rows, out_cols, Nd, out, ld_out);
    TC_KCHECK(h);
    return 0;
}
static int tc_colsum(dppo_handle* h, cudaStream_t s, const bf16* D, int N, int ncols, float* part, float* out) {
    int nb = 2 * h->sm_count; if (nb > (N + 63) / 64) nb = (N + 63) / 64; if (nb < 1) nb = 1;
    int rpb = (N + nb - 1) / nb; nb = (N + rpb - 1) / rpb;
    tc_colsum_kernel<<<nb, 256, 0, s>>>(D, N, ncols, rpb, part); TC_KCHECK(h);
    reduce_partials_kernel<<<tc_nblk(ncols, 256), 256, 0, s>>>(part, nb, (size_t)ncols, (size_t)ncols, out, 1.f); TC_KCHECK(h);
    return 0;
}
static size_t tc_part_floats(const dppo_handle* h, int H) {
    size_t a = (size_t)64 * H * 256, b = (size_t)2 * h->sm_count * H;     // generous: splits <= 64 on [H][<=256-wide share]
    size_t c = (size_t)h->sm_count * 128 * 256;                            // one 128x256 fp32 tile per CTA
    size_t m = a > b ? a : b;
    return m > c ? m : c;
}
// fused backward chain of one net (dv, dh1, du) + its bias column sums
static int tc_mlp_backward_dx(dppo_handle* h, cudaStream_t s, const TcMlp& m, const bf16* doutb, int N, float* part, float* gnet, size_t ob1, size_t ob2) {
    const int H = m.H;
    const int grid = fc::chain_grid(h, N);
    float* cpart = m.cpart ? m.cpart : part;                   // [grid][2][H]; `part` is consumed before anything reuses it
    DPPO_TRY(fc_bwd(h, s, m.net == DPPO_NET_CRITIC ? fc_critic_net(h) : fc_actor_net(h, m.net), doutb, N, m.m0, m.m1, m.pre0, m.pre1,
                    m.dv, m.dh1, m.du, cpart));
    if (!m.cpart) {   // slot 0 = column sums of dv (db2), slot 1 = of dh1 (db1)
        tc_reduce_cols_kernel<<<tc_nblk(2 * H, 8), 256, 0, s>>>(cpart, grid, (size_t)2 * H, 2 * H, gnet + ob2, H, gnet + ob1); TC_KCHECK(h);
    }
    return 0;
}
// the five weight-gradient products of one net as grouped-GEMM problems (outputs accumulate atomically); the narrow layer-0
// products are handed over as du^T h0 / dv^T h0 (transposed output)
static void tc_mlp_dw_pair_descs(const TcMlp& m, const bf16* doutb, int N, float* gnet, size_t ow1, size_t ow2, size_t ow3, float* dw0, tcp::PairDesc* d) {
    const int H = m.H, KP0 = m.KP0; const double r = (double)N;
    d[0] = tcp::PairDesc{m.a1, H, m.dv, H, gnet + ow2, H, H, H, 0, 2.0 * r * H * H};
    d[1] = tcp::PairDesc{m.a0, H, m.dh1, H, gnet + ow1, H, H, H, 0, 2.0 * r * H * H};
    d[2] = tcp::PairDesc{m.du, H, m.h0, KP0, dw0, H, KP0, H, 1, 2.0 * r * m.din * H};
    d[3] = tcp::PairDesc{m.dv, H, m.h0, KP0, dw0, H, KP0, H, 1, 0.0};                 // residual path: not algorithmic work
    d[4] = tcp::PairDesc{m.v, H, doutb, 64, gnet + ow3, H, m.NO, m.NO, 0, 2.0 * r * H * m.NO};
}
// backward of the residual MLP from doutb [N][64] (bf16, zero padded).  Writes gradients of W1,b1,W2,b2,W3 into gnet
// at the given offsets and dW0 (in h0 row order) into dw0 [KP0][H].
static int tc_mlp_backward(dppo_handle* h, cudaStream_t s, const TcMlp& m, const bf16* doutb, int N, float* part,
                           float* gnet, size_t ow1, size_t ob1, size_t ow2, size_t ob2, size_t ow3, float* dw0) {
    const int H = m.H, KP0 = m.KP0; const TcNetW& W = *m.W;
    if (m.fused) {
        // one launch: dv, dh1 and the non-residual part of du; the residual path joins in dW0 = h0^T du + h0^T dv
        DPPO_TRY(tc_mlp_backward_dx(h, s, m, doutb, N, part, gnet, ob1, ob2));
        if (!h->deterministic) {   // all five weight-gradient products in one grouped launch
            tcp::PairDesc pd[5];
            tc_mlp_dw_pair_descs(m, doutb, N, gnet, ow1, ow2, ow3, dw0, pd);
            return tcp::launch_group_pair(h, s, pd, 5, N);
        }
        DPPO_TRY(tc_dw(h, s, m.v, H, doutb, 64, N, part, gnet + ow3, H, m.NO, m.NO));
        DPPO_TRY(tc_dw(h, s, m.a1, H, m.dv, H, N, part, gnet + ow2, H, H, H));
        DPPO_TRY(tc_dw(h, s, m.a0, H, m.dh1, H, N, part, gnet + ow1, H, H, H));
        DPPO_TRY(tc_dw(h, s, m.h0, KP0, m.du, H, N, part, dw0, KP0, H, H, m.dv, m.din));
        return 0;
    }
    // dv = dout W3^T
    tc::Gemm g = gemm_of(opK(doutb, N, 64, 64), opK(W.w3p, H, 64, 128), N, H);
    g.epi.out_bf16 = m.dv; g.epi.ld_bf16 = H;
    DPPO_TRY(tc_run(h, s, g));
    // dh1 = (dv W2^T) * act'(h1)
    g = gemm_of(opK(m.dv, N, H, H), opK(W.w2w0, H, H, H), N, H);
    g.epi.mask = m.act1 == 2 ? m.pre1 : m.a1; g.epi.ldmask = H; g.epi.mask_mode = m.act1;
    g.epi.out_bf16 = m.dh1; g.epi.ld_bf16 = H;
    DPPO_TRY(tc_run(h, s, g));
    // du = (dh1 W1^T) * act'(u) + dv
    g = gemm_of(opK(m.dh1, N, H, H), opK(W.w1, H, H, H), N, H);
    g.epi.mask = m.act1 == 2 ? m.pre0 : m.a0; g.epi.ldmask = H; g.epi.mask_mode = m.act1;
    g.epi.add = m.dv; g.epi.ldadd = H; g.epi.out_bf16 = m.du; g.epi.ld_bf16 = H;
    DPPO_TRY(tc_run(h, s, g));
    // weight gradients
    DPPO_TRY(tc_dw(h, s, m.v, H, doutb, 64, N, part, gnet + ow3, H, m.NO, m.NO));
    DPPO_TRY(tc_dw(h, s, m.a1, H, m.dv, H, N, part, gnet + ow2, H, H, H));
    DPPO_TRY(tc_dw(h, s, m.a0, H, m.dh1, H, N, part, gnet + ow1, H, H, H));
    DPPO_TRY(tc_dw(h, s, m.h0, KP0, m.du, H, N, part, dw0, KP0, H, H, nullptr, m.din));
    // bias gradients of block.l1 / block.l2 (the input-layer bias comes out of dw0's constant rows)
    DPPO_TRY(tc_colsum(h, s, m.dv, N, H, part, gnet + ob2));
    DPPO_TRY(tc_colsum(h, s, m.dh1, N, H, part, gnet + ob1));
    return 0;
}

static void tc_actor_mlp(const dppo_handle* h, int net, TcMlp& m) {
    const Geom& g = h->g; const float* w = h->net_w[net];
    m.W = &h->tc->net[net]; m.H = g.H; m.NO = g.A; m.act1 = h->cfg.actor_act + 1; m.KP0 = h->tc->KP0;
    m.fused = fc_ok(h) ? 1 : 0; m.net = net; m.din = g.Din; m.cpart = nullptr;
    m.b0 = nullptr; m.b1 = w + g.ao.b1; m.b2 = w + g.ao.b2; m.b3 = w + g.ao.b3;
}
static void tc_critic_mlp(const dppo_handle* h, TcMlp& m) {
    const Geom& g = h->g; const float* w = h->net_w[DPPO_NET_CRITIC];
    m.W = &h->tc->net[DPPO_NET_CRITIC]; m.H = g.Hc; m.NO = 1; m.act1 = h->cfg.critic_act + 1; m.KP0 = h->tc->KP0;
    m.fused = fc_critic_ok(h) ? 1 : 0; m.net = DPPO_NET_CRITIC; m.din = g.Do; m.cpart = nullptr;
    m.b0 = w + g.co.bin; m.b1 = w + g.co.b1; m.b2 = m.W->bias2; m.b3 = w + g.co.b3;
}

// ------------------------------------------------------------------ forward-only: eps[N][A] = actor(x, t, obs)
// the buffers tc_actor_forward appends for N rows: h0, and the layer activations unless the fused chain runs the forward
static bf16* tc_actor_forward_take(dppo_handle* h, int net, int N, TcMlp& m) {
    tc_actor_mlp(h, net, m);
    bf16* h0 = ws_take<bf16>(h, (size_t)N * h->tc->KP0);
    if (!fc_ok(h)) tc_mlp_take(h, N, m, false);
    m.h0 = h0;
    return h0;
}
static int tc_actor_forward(dppo_handle* h, cudaStream_t s, int net, const float* x, const float* obs, int obs_div, int N,
                            const int* trow, int tconst, float* eps) {
    const Geom& g = h->g; const int KP0 = h->tc->KP0;
    // the caller may hold workspace pointers (eps, trow) below ws.used: only append
    const size_t mark = h->ws.used;
    TcMlp m; bf16* h0;
    DPPO_TRY(ws_append(h->ws, [&] { h0 = tc_actor_forward_take(h, net, N, m); }));
    m.out = eps;
    tc_pack_h0_kernel<<<tc_nblk((size_t)N * (KP0 / 8), 256), 256, 0, s>>>(x, obs, trow, tconst, N, g.A, g.Do, g.T, KP0, obs_div, h0);
    TC_KCHECK(h);
    const int r = fc_ok(h) ? fc_actor_infer(h, s, net, h0, N, fc::FINAL_EPS, eps, nullptr, nullptr, nullptr, nullptr) : tc_mlp_forward(h, s, m, N);
    h->ws.used = mark;
    return r;
}
static int tc_value(dppo_handle* h, cudaStream_t s, const float* obs, int N, float* v) {
    const Geom& g = h->g; const int KP0 = h->tc->KP0;
    TcMlp m; tc_critic_mlp(h, m);
    bf16* h0;
    DPPO_TRY(ws_layout(h->ws, s, [&] { h0 = ws_take<bf16>(h, (size_t)N * KP0); tc_mlp_take(h, N, m, false); }));
    m.h0 = h0; m.out = v;
    // the critic only reads the obs block (the x / one-hot rows of its W0 are zero)
    tc_pack_h0_kernel<<<tc_nblk((size_t)N * (KP0 / 8), 256), 256, 0, s>>>(nullptr, obs, nullptr, -1, N, g.A, g.Do, g.T, KP0, 1, h0);
    TC_KCHECK(h);
    if (fc_critic_ok(h)) return fc_infer(h, s, fc_critic_net(h), h0, N, fc::FINAL_EPS, v, nullptr, nullptr, nullptr, nullptr);
    return tc_mlp_forward(h, s, m, N);
}

// ------------------------------------------------------------------ gradients of the PPO / pre-train losses
static int colsum(dppo_handle* h, cudaStream_t s, const float* D, int ld, int N, int ncols, const int* seg, int nseg,
                  float* part, float* out);   // dppo_api.cu

// The layer-0 gradients of both tensor modes (dw0 [KP0][H] in h0's row order) into the flat gradient as separate launches: the actor's
// rows [A+Do, A+Do+T) are the per-t column sums of du (the gradient of the bt table, through the time backward) and its x / obs rows
// are dW_in; the critic's obs rows are its dW_in and the ones column collected its input-layer bias gradient.
// dw0c == nullptr: no critic (pre-training).  gr = [actor net's gradient (nA) | critic's].
static int tc_scatter_dw0(dppo_handle* h, cudaStream_t s, int net, const float* dw0a, const float* dw0c, float* gr) {
    const Geom& g = h->g;
    CUDA_TRY(launch_time_backward(h, s, net, dw0a + (size_t)(g.A + g.Do) * g.H, gr)); TC_KCHECK(h);
    unpack_dw0_kernel<<<tc_nblk((size_t)(g.A + g.Do) * g.H, 256), 256, 0, s>>>(dw0a, g.A, g.td, g.Do, g.H, gr + g.ao.win); TC_KCHECK(h);
    if (!dw0c) return 0;
    float* gc = gr + g.ao.n;
    unpack_dw0_kernel<<<tc_nblk((size_t)g.Do * g.Hc, 256), 256, 0, s>>>(dw0c + (size_t)g.A * g.Hc, 0, 0, g.Do, g.Hc, gc + g.co.win); TC_KCHECK(h);
    CUDA_TRY(cudaMemcpyAsync(gc + g.co.bin, dw0c + (size_t)(g.A + g.Do + g.T) * g.Hc, g.Hc * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return 0;
}
// advantage statistics of the whole minibatch (diffusion_ppo.py:74-75) into h->scalars: computed (adv_std < 0) from adv [N] or, with
// iv != nullptr, from the rollout advantages through the index view; else the given ones
static int launch_adv_stats(dppo_handle* h, cudaStream_t s, const float* adv, const TcIdxView* iv, int N, float adv_mean, float adv_std) {
    if (adv_std < 0.f) adv_stats_kernel<<<1, 1024, 0, s>>>(iv ? iv->adv : adv, N, h->scalars, iv ? iv->flat : nullptr, iv ? iv->K : 1, iv ? iv->P : 0);
    else set_scalars_kernel<<<1, 1, 0, s>>>(h->scalars, adv_mean, adv_std);
    TC_KCHECK(h);
    return 0;
}
// The loss8 kernels (tc_ppo_loss8_kernel) read rows as float4: A % 4 == 0, A <= max_a (32 for LPR = 8, 128 for a warp per row) and the
// row arrays 16-byte aligned (the minibatch's prev / nxt / oldlogp, or the index view's chains / olp)
static bool loss8_ok(int A, int max_a, const void* p0, const void* p1, const void* p2 = nullptr) {
    return A % 4 == 0 && A <= max_a && (((uintptr_t)p0 | (uintptr_t)p1 | (uintptr_t)p2) & 15) == 0;
}
// the second stream of the overlapped tensor schedules and its three events (fork, join, the split-precision fold), made on first use
static int ensure_aux_stream(dppo_handle* h) {
    if (h->aux_stream) return 0;
    CUDA_TRY(cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 3; ++i) CUDA_TRY(cudaEventCreateWithFlags(&h->aux_ev[i], cudaEventDisableTiming));
    return 0;
}

// actor backward from deps [N][A] fp32 (+ its padded bf16 copy): fills gnet[0 : nA]
static int tc_actor_grads(dppo_handle* h, cudaStream_t s, int net, const TcMlp& m, const float* deps, const bf16* depsb, int N,
                          float* part, float* dw0, float* gnet) {
    const Geom& g = h->g;
    DPPO_TRY(tc_mlp_backward(h, s, m, depsb, N, part, gnet, g.ao.w1, g.ao.b1, g.ao.w2, g.ao.b2, g.ao.w3, dw0));
    if (deps) DPPO_TRY(colsum(h, s, deps, g.A, N, g.A, nullptr, 1, part, gnet + g.ao.b3));   // else: the loss kernel already reduced it
    return tc_scatter_dw0(h, s, net, dw0, nullptr, gnet);
}

// PPODiffusion.c_loss + tape.gradient (diffusion_ppo.py:32-132, train_ppo_diffusion_agent.py:340-346) on the tensor path,
// as begin / chunk x C / finish so that the host-buffer entry point can overlap the H2D copy of chunk c+1 with the
// compute of chunk c (rows are independent; every gradient piece accumulates: dW by red.global.add, bias column sums
// and metric sums as per-block partials reduced once in finish).  Leaves [actor_ft grads | critic grads | 8 metrics]
// in h->grads.  The deterministic mode (fixed-order split-K reduction) supports a single chunk only.
struct TcPpoPlan {
    int N, nchunks, chunk_rows, lead_rows, blocks_done, max_blocks;
    int full_rows, rows_done, dw_done, dw_flush_chunk;
    TcIdxView idx;                                        // idx.flat != nullptr: the (single) chunk reads the rollout buffers through flat indices   // multi-chunk pipeline: per-row buffers hold ALL rows, dW runs in (at most) two launches
    int64_t N_global;
    float *part, *dw0a, *dw0c, *colb3, *cpa, *cpc;
    double* bsum;
    TcMlp ma, mc;
    bf16 *h0, *depsb, *dvalb; float *eps, *val;
    PpoHyper hp;
};
static TcPpoPlan& tc_plan(dppo_handle* h) { if (!h->tc->plan) { h->tc->plan = new TcPpoPlan(); memset(h->tc->plan, 0, sizeof(TcPpoPlan)); } return *h->tc->plan; }
static void tc_plan_free(dppo_handle* h) { if (h->tc && h->tc->plan) { delete h->tc->plan; h->tc->plan = nullptr; } }

// chunk_rows <= 0 or >= N: one chunk
// lead_rows > 0: the host pipeline starts with a shorter chunk of that many rows (its copy lands early), then chunk_rows-sized ones
static int tc_ppo_begin(dppo_handle* h, cudaStream_t s, int N, int chunk_rows, int64_t N_global, int lead_rows = 0) {
    const Geom& g = h->g; const int KP0 = h->tc->KP0;
    const size_t nA = g.ao.n, nC = g.co.n;
    TcPpoPlan& P = tc_plan(h);
    if (h->deterministic || chunk_rows <= 0 || chunk_rows >= N) chunk_rows = N;
    chunk_rows = round_up(chunk_rows, 128);
    if (lead_rows <= 0 || lead_rows >= chunk_rows || chunk_rows >= N) lead_rows = 0;
    const int nchunks = lead_rows ? 1 + (N - lead_rows + chunk_rows - 1) / chunk_rows : (N + chunk_rows - 1) / chunk_rows;
    P.N = N; P.nchunks = nchunks; P.N_global = N_global; P.blocks_done = 0;
    memset(&P.idx, 0, sizeof(P.idx));
    P.chunk_rows = chunk_rows; P.lead_rows = lead_rows;
    // More than one chunk (host pipeline): every per-row buffer holds all N rows and chunk c works on its own row range, so that
    // the weight-gradient GEMMs need not run once per chunk (each launch pays a full set of output-tile reductions): one launch
    // covers the chunks of the first half while the rest is still on the link, one covers the remainder.
    P.full_rows = nchunks > 1 ? 1 : 0; P.rows_done = 0; P.dw_done = 0; P.dw_flush_chunk = nchunks / 2 - 1;
    const int NC = P.full_rows ? N : (P.chunk_rows < N ? P.chunk_rows : N);
    P.max_blocks = tc_nblk(N, LOSS8_ROWS) + nchunks;
    const size_t n_cpa = (size_t)nchunks * h->sm_count * 2 * g.H, n_cpc = (size_t)nchunks * h->sm_count * 2 * g.Hc;
    tc_actor_mlp(h, DPPO_NET_ACTOR_FT, P.ma); tc_critic_mlp(h, P.mc);
    DPPO_TRY(ws_layout(h->ws, s, [&] {
        P.h0 = ws_take<bf16>(h, (size_t)NC * KP0);
        tc_mlp_take(h, NC, P.ma, true); tc_mlp_take(h, NC, P.mc, true);
        P.eps = ws_take<float>(h, (size_t)NC * g.A); P.val = ws_take<float>(h, NC);
        P.depsb = ws_take<bf16>(h, (size_t)NC * 64); P.dvalb = ws_take<bf16>(h, (size_t)NC * 64);
        P.part = ws_take<float>(h, tc_part_floats(h, g.H));
        P.bsum = ws_take<double>(h, (size_t)P.max_blocks * 5);
        P.colb3 = ws_take<float>(h, (size_t)P.max_blocks * (g.A + 1));
        // the four accumulators below are adjacent so that one memset clears them
        P.dw0a = ws_take<float>(h, (size_t)KP0 * g.H); P.dw0c = ws_take<float>(h, (size_t)KP0 * g.Hc);
        P.cpa = ws_take<float>(h, n_cpa); P.cpc = ws_take<float>(h, n_cpc);
    }));
    const size_t acc_bytes = (size_t)((char*)(P.cpc + n_cpc) - (char*)P.dw0a);
    P.ma.h0 = P.h0; P.mc.h0 = P.h0; P.ma.out = P.eps; P.mc.out = P.val;
    const bool defer = P.ma.fused && P.mc.fused && !h->deterministic;
    if (!defer && nchunks > 1) DPPO_FAIL(-7, "tc_ppo_begin: chunked accumulation needs the fused chain kernels");
    if (!h->deterministic) {   // the dW GEMMs accumulate atomically into the gradient buffers
        CUDA_TRY(cudaMemsetAsync(h->grads, 0, (nA + nC) * sizeof(float), s));
        CUDA_TRY(cudaMemsetAsync(P.dw0a, 0, acc_bytes, s));
    }
    P.hp = ppo_hyper(h, N_global);
    return 0;
}
// advantage statistics for the whole minibatch: given, or computed from the device array
static int tc_ppo_adv_stats(dppo_handle* h, cudaStream_t s, const float* advantages_all, int N, float adv_mean, float adv_std) {
    // only the loss kernel reads the statistics: with the two-stream schedule they are computed on the second stream, next to
    // pack_h0 and the forward chains (the join in front of the loss kernel orders them)
    TcPpoPlan& P = tc_plan(h);
    cudaStream_t st = s;
    if (P.ma.fused && P.mc.fused && !h->deterministic && !h->prof_on) {
        DPPO_TRY(ensure_aux_stream(h));
        CUDA_TRY(cudaEventRecord(h->aux_ev[0], s)); CUDA_TRY(cudaStreamWaitEvent(h->aux_stream, h->aux_ev[0], 0));
        st = h->aux_stream;
    }
    return launch_adv_stats(h, st, advantages_all, P.idx.flat ? &P.idx : nullptr, N, adv_mean, adv_std);
}
// chunk size of the host pipeline: half waves of 128-row tiles (one tile per SM pair member), at most 7 chunks (+ the short lead
// chunk); 0 = do not chunk.  Every chunk costs a start-up / drain of the four persistent chain kernels (~10 us each), so the
// pipeline recovers only part of the copy time; half-wave chunks with the weight-gradient GEMMs deferred measured best.
static int tc_ppo_pipeline_chunk_rows(const dppo_handle* h, int N) {
    const int wave = h->sm_count * 128;
    if (N < 2 * wave) return 0;
    int c = wave / 2;
    while ((N + c - 1) / c > 7) c += wave / 2;
    return c;
}
// rows [r0, r0 + n) of the minibatch; all pointers already point at row r0
static int tc_ppo_chunk(dppo_handle* h, cudaStream_t s, int chunk, const float* obs, const float* prev, const float* nxt, const int32_t* inds,
                        const float* returns, const float* oldvalues, const float* advantages, const float* oldlogp, int n) {
    const Geom& g = h->g; const int KP0 = h->tc->KP0;
    const size_t nA = g.ao.n;
    TcPpoPlan& P = tc_plan(h);
    if (n < 1 || n > P.chunk_rows || chunk < 0 || chunk >= P.nchunks) DPPO_FAIL(-1, "tc_ppo_chunk: bad chunk");
    const TcIdxView iv = P.idx;
    const bool loss8 = iv.flat ? loss8_ok(g.A, 32, iv.chains, iv.olp) : loss8_ok(g.A, 32, prev, nxt, oldlogp);
    if (iv.flat && (!loss8 || P.nchunks != 1)) DPPO_FAIL(-1, "tc_ppo_chunk: the index-driven minibatch needs A % 4 == 0, aligned buffers and a single chunk");
    const int nlb = loss8 ? tc_nblk(n, LOSS8_ROWS) : tc_nblk(n, 128);
    if (P.blocks_done + nlb > P.max_blocks) DPPO_FAIL(-1, "tc_ppo_chunk: partial-sum buffers exhausted");
    const bool defer = P.ma.fused && P.mc.fused && !h->deterministic;
    P.ma.cpart = defer ? P.cpa + (size_t)chunk * h->sm_count * 2 * g.H : nullptr;
    P.mc.cpart = defer ? P.cpc + (size_t)chunk * h->sm_count * 2 * g.Hc : nullptr;
    const size_t r0 = P.full_rows ? (size_t)P.rows_done : 0;          // this chunk's rows inside the per-row buffers
    if (r0 + (size_t)n > (size_t)P.N) DPPO_FAIL(-1, "tc_ppo_chunk: more rows than planned");
    const TcMlp ma = tc_mlp_at(P.ma, r0), mc = tc_mlp_at(P.mc, r0);
    bf16* const depsb = P.depsb + r0 * 64; bf16* const dvalb = P.dvalb + r0 * 64;
    // h0 straight from (prev, obs, K-1-inds): tconst = -(K) flags "t = K-1-trow[r]"
    if (iv.flat)
        tc_pack_h0_kernel<<<tc_nblk((size_t)n * (KP0 / 8), 256), 256, 0, s>>>(iv.chains, iv.obs, nullptr, 0, n, g.A, g.Do, g.T, KP0, 1, P.h0 + r0 * KP0, 0,
                                                                                iv.flat, iv.K, iv.P, iv.bad);
    else
        tc_pack_h0_kernel<<<tc_nblk((size_t)n * (KP0 / 8), 256), 256, 0, s>>>(prev, obs, inds, -g.K, n, g.A, g.Do, g.T, KP0, 1, P.h0 + r0 * KP0);
    TC_KCHECK(h);
    // The actor and the critic chains are independent persistent kernels whose last wave leaves a third of the SMs idle
    // (391 row tiles on 148 SMs): the critic chain goes to a second stream so that its CTAs fill the actor chain's tail.
    // (not while the per-kernel profile is on: its event brackets are meant to time each kernel running alone)
    const bool overlap = defer && !h->prof_on;
    if (overlap) DPPO_TRY(ensure_aux_stream(h));
    auto fork = [&]() -> int { CUDA_TRY(cudaEventRecord(h->aux_ev[0], s)); CUDA_TRY(cudaStreamWaitEvent(h->aux_stream, h->aux_ev[0], 0)); return 0; };
    auto join = [&]() -> int { CUDA_TRY(cudaEventRecord(h->aux_ev[1], h->aux_stream)); CUDA_TRY(cudaStreamWaitEvent(s, h->aux_ev[1], 0)); return 0; };
    if (overlap) DPPO_TRY(fork());
    DPPO_TRY(tc_mlp_forward(h, s, ma, n));
    DPPO_TRY(tc_mlp_forward(h, overlap ? h->aux_stream : s, mc, n));
    if (overlap) DPPO_TRY(join());
    if (loss8)
        tc_ppo_loss8_kernel<<<nlb, 256, 0, s>>>(prev, nxt, ma.out, inds, returns, oldvalues, advantages, oldlogp, mc.out,
                                               h->scalars, h->sched, P.hp, n, depsb, dvalb, P.bsum + (size_t)P.blocks_done * 5,
                                               P.colb3 + (size_t)P.blocks_done * (g.A + 1), iv);
    else
        tc_ppo_loss_kernel<<<nlb, 128, 0, s>>>(prev, nxt, ma.out, inds, returns, oldvalues, advantages, oldlogp, mc.out,
                                              h->scalars, h->sched, P.hp, n, depsb, dvalb, P.bsum + (size_t)P.blocks_done * 5,
                                              P.colb3 + (size_t)P.blocks_done * (g.A + 1));
    TC_KCHECK(h);
    P.blocks_done += nlb;
    if (defer) {
        // both backward chains, then ONE grouped launch with the ten weight-gradient products of actor and critic
        if (overlap) DPPO_TRY(fork());
        DPPO_TRY(tc_mlp_backward_dx(h, s, ma, depsb, n, P.part, h->grads, g.ao.b1, g.ao.b2));
        DPPO_TRY(tc_mlp_backward_dx(h, overlap ? h->aux_stream : s, mc, dvalb, n, P.part, h->grads + nA, g.co.b1, g.co.b2));
        if (overlap) DPPO_TRY(join());
        P.rows_done += n;
        // weight gradients over the rows accumulated since the last launch: every chunk (single-chunk call), or at the flush chunk and the end
        if (P.full_rows && chunk != P.dw_flush_chunk && P.rows_done < P.N) return 0;
        const size_t d0 = P.full_rows ? (size_t)P.dw_done : r0;
        const int dn = (int)((P.full_rows ? (size_t)P.rows_done : r0 + (size_t)n) - d0);
        const TcMlp da = tc_mlp_at(P.ma, d0), dc = tc_mlp_at(P.mc, d0);
        const bf16* const dd = P.depsb + d0 * 64; const bf16* const dvd = P.dvalb + d0 * 64;
        P.dw_done = P.rows_done;
        tcp::PairDesc pd[10];
        tc_mlp_dw_pair_descs(da, dd, dn, h->grads, g.ao.w1, g.ao.w2, g.ao.w3, P.dw0a, pd);
        tc_mlp_dw_pair_descs(dc, dvd, dn, h->grads + nA, g.co.w1, g.co.w2, g.co.w3, P.dw0c, pd + 5);
        return tcp::launch_group_pair(h, s, pd, 10, dn);
    }
    DPPO_TRY(tc_mlp_backward(h, s, ma, depsb, n, P.part, h->grads, g.ao.w1, g.ao.b1, g.ao.w2, g.ao.b2, g.ao.w3, P.dw0a));
    DPPO_TRY(tc_mlp_backward(h, s, mc, dvalb, n, P.part, h->grads + nA, g.co.w1, g.co.b1, g.co.w2, g.co.b2, g.co.w3, P.dw0c));
    P.rows_done += n;
    return 0;
}
// Everything between the weight-gradient GEMM and AdamW in one launch (tc_ppo_tail_kernel): metric sums, output-layer bias
// gradients from the loss kernel's column partials, hidden-layer bias gradients from the chains' per-row-block column sums
// (cpa / cpc: [rows][2][H], slot 0 = dv -> db2, slot 1 = dh1 -> db1), time-embedding backward, dW0 scatters, critic input bias.
static int tc_launch_tail(dppo_handle* h, cudaStream_t s, const double* bsum, int blocks_done, float inv_nglobal, float frac_local, const float* colb3,
                          const float* cpa, int rows_a, const float* cpc, int rows_c, const float* dw0a, const float* dw0c,
                          float* b2a_out = nullptr, float* b2c_out = nullptr) {   // b2*_out: where the slot-0 sums go instead of the b2 gradients
                                                                                    // (programs that never form dv leave slot 0 unwritten)
    const Geom& g = h->g;
    const size_t nA = g.ao.n, nC = g.co.n;
    float* gr = h->grads;
    const float* w = h->net_w[DPPO_NET_ACTOR_FT]; const ActorDerived& d = h->ad[DPPO_NET_ACTOR_FT];
    const size_t sm = time_backward_smem(g);
    if (sm > 160 * 1024) DPPO_FAIL(-7, "tc_launch_tail: time_dim x denoising_steps too large");
    static bool attr_set_dev[64] = {};      // function attributes are per device
    bool& attr_set = attr_set_dev[h->device & 63];
    if (!attr_set) { CUDA_TRY(cudaFuncSetAttribute(tc_ppo_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024)); attr_set = true; }
    TcTailArgs a;
    const int nthr = 512, wpb = nthr / 32;
    const bool wide = rows_a >= 256;         // many partial rows (plane GEMM epilogues): the coalesced 32-columns-per-block reduction
    const int cpb = wide ? 32 : wpb;
    const bool wide3 = blocks_done >= 256;
    a.wide = wide ? 1 : 0; a.wide3 = wide3 ? 1 : 0;
    const int nb[8] = {1, tc_nblk(g.A + 1, wide3 ? 32 : wpb), tc_nblk(2 * g.H, cpb), tc_nblk(2 * g.Hc, cpb), time_backward_grid(g),
                       tc_nblk((size_t)(g.A + g.Do) * g.H, nthr), tc_nblk((size_t)g.Do * g.Hc, nthr), tc_nblk(g.Hc, nthr)};
    a.first[0] = 0;
    for (int r = 0; r < 8; ++r) a.first[r + 1] = a.first[r] + nb[r];
    a.bsum = bsum; a.blocks_done = blocks_done; a.inv_nglobal = inv_nglobal; a.frac_local = frac_local; a.metrics = gr + nA + nC;
    a.colb3 = colb3; a.ncol3 = g.A + 1; a.b3a = gr + g.ao.b3; a.split3 = g.A; a.b3c = gr + nA + g.co.b3;
    a.cpa = cpa; a.rows_a = rows_a; a.HA = g.H; a.b2a = b2a_out ? b2a_out : gr + g.ao.b2; a.b1a = gr + g.ao.b1;
    a.cpc = cpc; a.rows_c = rows_c; a.HC = g.Hc; a.b2c = b2c_out ? b2c_out : gr + nA + g.co.b2; a.b1c = gr + nA + g.co.b1;
    a.w = w; a.ao = g.ao; a.A = g.A; a.td = g.td; a.T = g.T; a.Do = g.Do;
    a.Gt = dw0a + (size_t)(g.A + g.Do) * g.H; a.sinemb = d.sinemb; a.thpre = d.thpre; a.temb = d.temb; a.dte = d.dte; a.gr = gr;
    a.dw0a = dw0a; a.gwin_a = gr + g.ao.win; a.dw0c_obs = dw0c + (size_t)g.A * g.Hc; a.gwin_c = gr + nA + g.co.win;
    a.dw0c_bias = dw0c + (size_t)(g.A + g.Do + g.T) * g.Hc; a.gbin_c = gr + nA + g.co.bin;
    CUDA_TRY(launch_pdl(tc_ppo_tail_kernel, dim3(a.first[8]), dim3(nthr), sm, s, a)); TC_KCHECK(h);
    return 0;
}
static int tc_ppo_finish(dppo_handle* h, cudaStream_t s) {
    const Geom& g = h->g;
    const size_t nA = g.ao.n, nC = g.co.n;
    TcPpoPlan& P = tc_plan(h);
    float* gr = h->grads;
    const bool defer = P.ma.fused && P.mc.fused && !h->deterministic;
    if (defer) return tc_launch_tail(h, s, P.bsum, P.blocks_done, P.hp.inv_nglobal, (float)((double)P.N / (double)P.N_global), P.colb3,
                                     P.cpa, P.nchunks * h->sm_count, P.cpc, P.nchunks * h->sm_count, P.dw0a, P.dw0c);
    ppo_metrics_kernel<<<1, 256, 0, s>>>(P.bsum, P.blocks_done, P.hp.inv_nglobal, (float)((double)P.N / (double)P.N_global), gr + nA + nC); TC_KCHECK(h);
    // output-layer bias gradients = column sums of the seeds (per-block partials from the loss kernel)
    tc_reduce_cols_kernel<<<tc_nblk(g.A + 1, 8), 256, 0, s>>>(P.colb3, P.blocks_done, (size_t)(g.A + 1), g.A + 1, gr + g.ao.b3, g.A, gr + nA + g.co.b3); TC_KCHECK(h);
    return tc_scatter_dw0(h, s, DPPO_NET_ACTOR_FT, P.dw0a, P.dw0c, gr);
}
static int tc_ppo_step(dppo_handle* h, cudaStream_t s, const float* obs, const float* prev, const float* nxt, const int32_t* inds,
                       const float* returns, const float* oldvalues, const float* advantages, const float* oldlogp,
                       int N, int64_t N_global, float adv_mean, float adv_std) {
    DPPO_TRY(tc_ppo_begin(h, s, N, 0, N_global));
    DPPO_TRY(tc_ppo_adv_stats(h, s, advantages, N, adv_mean, adv_std));
    DPPO_TRY(tc_ppo_chunk(h, s, 0, obs, prev, nxt, inds, returns, oldvalues, advantages, oldlogp, N));
    return tc_ppo_finish(h, s);
}

// the same update with the minibatch given as flat (rollout row, denoising index) indices into the resident rollout buffers
static bool tc_ppo_indexed_ok(const dppo_handle* h, const TcIdxView& v) {
    return loss8_ok(h->g.A, 32, v.chains, v.olp) && !h->deterministic && fc_ok(h) && fc_critic_ok(h);
}
static int tc_ppo_step_indexed(dppo_handle* h, cudaStream_t s, const TcIdxView& view, int N, int64_t N_global, float adv_mean, float adv_std) {
    DPPO_TRY(tc_ppo_begin(h, s, N, 0, N_global));
    tc_plan(h).idx = view;
    DPPO_TRY(tc_ppo_adv_stats(h, s, nullptr, N, adv_mean, adv_std));
    DPPO_TRY(tc_ppo_chunk(h, s, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, N));
    tc_plan(h).idx.flat = nullptr;
    return tc_ppo_finish(h, s);
}

// DiffusionModel.c_loss / p_losses (diffusion.py:179-202) + tape.gradient on the tensor path: loss -> h->grads[nA],
// gradients -> h->grads[0 : nA]
static int tc_pretrain_grads(dppo_handle* h, cudaStream_t s, const float* actions, const float* obs, int N, int64_t N_global,
                             int64_t row_offset, const int32_t* t_in, const float* noise_in, uint64_t seed, uint64_t offset) {
    const Geom& g = h->g; const int KP0 = h->tc->KP0;
    const size_t nA = g.ao.n; float* gr = h->grads;
    const size_t ne = (size_t)N * g.A;
    const int nlb = tc_nblk(ne, 256);
    TcMlp ma; tc_actor_mlp(h, DPPO_NET_ACTOR, ma);
    bf16 *h0, *depsb; float *eps, *deps, *noise, *xn, *part, *dw0; int* trow; double* bsum;
    DPPO_TRY(ws_layout(h->ws, s, [&] {
        h0 = ws_take<bf16>(h, (size_t)N * KP0);
        tc_mlp_take(h, N, ma, true);
        eps = ws_take<float>(h, ne); deps = ws_take<float>(h, ne); noise = ws_take<float>(h, ne); xn = ws_take<float>(h, ne);
        trow = ws_take<int>(h, N);
        depsb = ws_take<bf16>(h, (size_t)N * 64);
        part = ws_take<float>(h, tc_part_floats(h, g.H));
        dw0 = ws_take<float>(h, (size_t)KP0 * g.H);
        bsum = ws_take<double>(h, nlb);
    }));
    ma.h0 = h0; ma.out = eps;
    if (!h->deterministic) {
        CUDA_TRY(cudaMemsetAsync(gr, 0, nA * sizeof(float), s));
        CUDA_TRY(cudaMemsetAsync(dw0, 0, (size_t)KP0 * g.H * sizeof(float), s));
    }
    pretrain_prep_kernel<<<tc_nblk(ne, 256), 256, 0, s>>>(actions, t_in, noise_in, N, g.A, g.T, h->sched, seed, offset, row_offset, trow, noise, xn); TC_KCHECK(h);
    tc_pack_h0_kernel<<<tc_nblk((size_t)N * (KP0 / 8), 256), 256, 0, s>>>(xn, obs, trow, 0, N, g.A, g.Do, g.T, KP0, 1, h0); TC_KCHECK(h);
    DPPO_TRY(tc_mlp_forward(h, s, ma, N));
    const float scale = 1.0f / ((float)N_global * (float)g.A);
    mse_loss_kernel<<<nlb, 256, 0, s>>>(eps, noise, ne, scale, deps, bsum); TC_KCHECK(h);
    sum_blocks_kernel<<<1, 256, 0, s>>>(bsum, nlb, scale, gr + nA); TC_KCHECK(h);
    tc_pad64_kernel<<<tc_nblk((size_t)N * 8, 256), 256, 0, s>>>(deps, N, g.A, depsb); TC_KCHECK(h);
    DPPO_TRY(tc_actor_grads(h, s, DPPO_NET_ACTOR, ma, deps, depsb, N, part, dw0, gr));
    return 0;
}
