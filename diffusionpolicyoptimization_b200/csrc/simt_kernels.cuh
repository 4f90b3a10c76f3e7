// fp32 CUDA-core kernels: the strict-parity path (DPPO_PREC_FP32) and everything element-wise.
#pragma once
#include "common.cuh"

// =====================================================================================
// SGEMM  C[M,N] = epi( aop(A)[M,K] * B[K,N] )      (fp32 FFMA, 128 x BN x 16 tiles, 256 threads)
//   A_KM : A is stored [K][lda] (reduction index outermost; the dW = X^T D case)
//   B_NK : B is stored [N][ldb] (the dX = D W^T case, W kept [in,out])
//   split-K over gridDim.z writes partial sums to C + z*cstride (no epilogue).
// =====================================================================================
struct GemmP {
    const float* A; int lda;
    const float* B; int ldb;
    float* C; int ldc;
    int M, N, K;
    int kchunk; size_t cstride;
    int vecA, vecB, vecC;             // 16-byte vector access allowed for that operand
    int aop;                          // 0 none, 1 relu, 2 mish applied to A on load
    const float* bias;                // [N]
    const float* btab; int ldbt;      // bias table [T][ldbt], row picked by trow[m] or tconst
    const int* trow; int tconst;
    const float* mask; int ldm; int mask_act;   // C *= act'(mask[m][n])
    const float* add; int ldadd;      // C += add[m][n]
};

template <bool A_KM, bool B_NK, int BN>
__global__ void __launch_bounds__(256, 2) sgemm_kernel(const GemmP p) {
    constexpr int BM = 128, BK = 16, TN = BN / 16;
    __shared__ __align__(16) float As[2][BK][BM + 4];
    __shared__ __align__(16) float Bs[2][BK][BN + 4];

    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int kbeg = blockIdx.z * p.kchunk;
    const int kend = min(p.K, kbeg + p.kchunk);
    float* __restrict__ C = p.C + (size_t)blockIdx.z * p.cstride;
    const float* __restrict__ A = p.A;
    const float* __restrict__ B = p.B;
    const int aop = p.aop;

    float acc[8][TN];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    float4 ra[2], rb[2];

    auto load_a = [&](int k0) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            int f = tid + j * 256;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (!A_KM) {
                int row = f >> 2, k = k0 + (f & 3) * 4, m = m0 + row;
                if (m < p.M) {
                    const float* src = A + (size_t)m * p.lda + k;
                    if (p.vecA) { if (k < kend) v = *reinterpret_cast<const float4*>(src); }
                    else {
                        if (k + 0 < kend) v.x = src[0];
                        if (k + 1 < kend) v.y = src[1];
                        if (k + 2 < kend) v.z = src[2];
                        if (k + 3 < kend) v.w = src[3];
                    }
                }
            } else {
                int k = k0 + (f >> 5), m = m0 + (f & 31) * 4;
                if (k < kend) {
                    const float* src = A + (size_t)k * p.lda + m;
                    if (p.vecA) { if (m < p.M) v = *reinterpret_cast<const float4*>(src); }
                    else {
                        if (m + 0 < p.M) v.x = src[0];
                        if (m + 1 < p.M) v.y = src[1];
                        if (m + 2 < p.M) v.z = src[2];
                        if (m + 3 < p.M) v.w = src[3];
                    }
                }
            }
            if (aop) { v.x = act_rt(v.x, aop); v.y = act_rt(v.y, aop); v.z = act_rt(v.z, aop); v.w = act_rt(v.w, aop); }
            ra[j] = v;
        }
    };
    auto store_a = [&](int buf) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            int f = tid + j * 256;
            if (!A_KM) {
                int row = f >> 2, kq = (f & 3) * 4;
                As[buf][kq + 0][row] = ra[j].x; As[buf][kq + 1][row] = ra[j].y;
                As[buf][kq + 2][row] = ra[j].z; As[buf][kq + 3][row] = ra[j].w;
            } else {
                int k = f >> 5, mq = (f & 31) * 4;
                *reinterpret_cast<float4*>(&As[buf][k][mq]) = ra[j];
            }
        }
    };
    constexpr int BF4 = BK * BN / 4;          // float4s in a B tile: 512 (BN=128) or 128 (BN=32)
    constexpr int BJ = (BF4 + 255) / 256;
    auto load_b = [&](int k0) {
#pragma unroll
        for (int j = 0; j < BJ; ++j) {
            int f = tid + j * 256;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (f < BF4) {
                if (!B_NK) {
                    int k = k0 + f / (BN / 4), n = n0 + (f % (BN / 4)) * 4;
                    if (k < kend) {
                        const float* src = B + (size_t)k * p.ldb + n;
                        if (p.vecB) { if (n < p.N) v = *reinterpret_cast<const float4*>(src); }
                        else {
                            if (n + 0 < p.N) v.x = src[0];
                            if (n + 1 < p.N) v.y = src[1];
                            if (n + 2 < p.N) v.z = src[2];
                            if (n + 3 < p.N) v.w = src[3];
                        }
                    }
                } else {
                    int nn = f >> 2, k = k0 + (f & 3) * 4, n = n0 + nn;
                    if (n < p.N) {
                        const float* src = B + (size_t)n * p.ldb + k;
                        if (p.vecB) { if (k < kend) v = *reinterpret_cast<const float4*>(src); }
                        else {
                            if (k + 0 < kend) v.x = src[0];
                            if (k + 1 < kend) v.y = src[1];
                            if (k + 2 < kend) v.z = src[2];
                            if (k + 3 < kend) v.w = src[3];
                        }
                    }
                }
            }
            rb[j] = v;
        }
    };
    auto store_b = [&](int buf) {
#pragma unroll
        for (int j = 0; j < BJ; ++j) {
            int f = tid + j * 256;
            if (f < BF4) {
                if (!B_NK) {
                    int k = f / (BN / 4), nq = (f % (BN / 4)) * 4;
                    *reinterpret_cast<float4*>(&Bs[buf][k][nq]) = rb[j];
                } else {
                    int nn = f >> 2, kq = (f & 3) * 4;
                    Bs[buf][kq + 0][nn] = rb[j].x; Bs[buf][kq + 1][nn] = rb[j].y;
                    Bs[buf][kq + 2][nn] = rb[j].z; Bs[buf][kq + 3][nn] = rb[j].w;
                }
            }
        }
    };

    const int nk = (kend - kbeg + BK - 1) / BK;
    if (nk > 0) {
        load_a(kbeg); load_b(kbeg);
        store_a(0); store_b(0);
    }
    __syncthreads();
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nk) { load_a(kbeg + (kt + 1) * BK); load_b(kbeg + (kt + 1) * BK); }
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float a[8], b[TN];
            float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
            float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][64 + ty * 4]);
            a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
            if constexpr (TN == 8) {
                float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
                float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][k][64 + tx * 4]);
                b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w;
                b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
            } else {
                float2 b0 = *reinterpret_cast<const float2*>(&Bs[buf][k][tx * 2]);
                b[0] = b0.x; b[1] = b0.y;
            }
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        if (kt + 1 < nk) { store_a(buf ^ 1); store_b(buf ^ 1); }
        __syncthreads();
    }

    // ---- epilogue
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (m >= p.M) continue;
        const float* btrow = nullptr;
        if (p.btab) { int t = p.trow ? p.trow[m] : p.tconst; btrow = p.btab + (size_t)t * p.ldbt; }
#pragma unroll
        for (int jb = 0; jb < TN; jb += (TN == 8 ? 4 : 2)) {
            constexpr int W = (TN == 8 ? 4 : 2);
            const int n = n0 + (TN == 8 ? (jb < 4 ? tx * 4 : 64 + tx * 4) : tx * 2);
            float v[W];
#pragma unroll
            for (int e = 0; e < W; ++e) {
                float x = acc[i][jb + e];
                int nn = n + e;
                if (nn < p.N) {
                    if (p.bias) x += p.bias[nn];
                    if (btrow) x += btrow[nn];
                    if (p.mask) x *= act_grad_rt(p.mask[(size_t)m * p.ldm + nn], p.mask_act);
                    if (p.add) x += p.add[(size_t)m * p.ldadd + nn];
                }
                v[e] = x;
            }
            float* dst = C + (size_t)m * p.ldc + n;
            if (W == 4 && p.vecC && n + 3 < p.N) {
                *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
                for (int e = 0; e < W; ++e) if (n + e < p.N) dst[e] = v[e];
            }
        }
    }
}

// out[i] = scale * sum_s partial[s*stride + i]   (deterministic split-K reduction)
__global__ void reduce_partials_kernel(const float* __restrict__ part, int S, size_t stride, size_t n,
                                       float* __restrict__ out, float scale) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = 0.f;
    for (int k = 0; k < S; ++k) s += part[(size_t)k * stride + i];
    out[i] = s * scale;
}

// =====================================================================================
// Derived tables of an actor: sinusoidal embedding -> time MLP -> per-t layer-0 bias, packed W_in
//   modules.py:10-15, mlp_diffusion.py:40-45,83-86.  grid = T blocks of H threads (H <= 1024).
// =====================================================================================
// bt16 (optional): the same table rounded to bf16, written straight into the time rows of the packed layer-0 operand
// w(i): parameter i of the actor's flat vector (WRead: as stored; the fused update of the split-precision mode passes the
// AdamW-updated values)
struct WRead { const float* __restrict__ p; __device__ __forceinline__ float operator()(size_t i) const { return p[i]; } };
template <class WF>
__device__ __forceinline__ void actor_prep_body(const int t, float* sm, const WF w, ActorOff o, int A, int td, int H,
                                  float* __restrict__ sinemb, float* __restrict__ thpre,
                                  float* __restrict__ temb, float* __restrict__ bt, __nv_bfloat16* __restrict__ bt16) {
    float* se = sm;            // [td]
    float* hp = se + td;       // [2td]
    float* te = hp + 2 * td;   // [td]
    const int tid = threadIdx.x;
    const int half = td / 2;
    if (tid < td) {
        int i = tid % half;
        float f = expf((float)i * -(logf(10000.f) / (float)(half - 1)));
        float e = (float)t * f;
        float v = tid < half ? sinf(e) : cosf(e);
        se[tid] = v; sinemb[t * td + tid] = v;
    }
    __syncthreads();
    if (tid < 2 * td) {
        float s = w(o.tb1 + tid);
        for (int j = 0; j < td; ++j) s = fmaf(se[j], w(o.tw1 + (size_t)j * 2 * td + tid), s);
        thpre[t * 2 * td + tid] = s;
        hp[tid] = mish_f(s);
    }
    __syncthreads();
    if (tid < td) {
        float s = w(o.tb2 + tid);
        for (int j = 0; j < 2 * td; ++j) s = fmaf(hp[j], w(o.tw2 + (size_t)j * td + tid), s);
        te[tid] = s; temb[t * td + tid] = s;
    }
    __syncthreads();
    for (int c = tid; c < H; c += blockDim.x) {
        float s = w(o.bin + c);
        for (int j = 0; j < td; ++j) s = fmaf(te[j], w(o.win + (size_t)(A + j) * H + c), s);
        bt[(size_t)t * H + c] = s;
        if (bt16) bt16[(size_t)t * H + c] = __float2bfloat16(s);
    }
}
__global__ void actor_prep_kernel(const float* __restrict__ w, ActorOff o, int A, int td, int H,
                                  float* __restrict__ sinemb, float* __restrict__ thpre,
                                  float* __restrict__ temb, float* __restrict__ bt) {
    extern __shared__ float sm[];
    actor_prep_body(blockIdx.x, sm, WRead{w}, o, A, td, H, sinemb, thpre, temb, bt, nullptr);
}
// w23[k][a] = sum_j W2[k][j] W3[j][a] (k < H), b23[a] = b3[a] + sum_j b2[j] W3[j][a] (the thread row k == H): products of the folded output
// layer (MLP / ResidualMLP of model/common/mlp.py: the last Dense follows the residual add without an activation)
__global__ void fold_output_kernel(const float* __restrict__ w2, const float* __restrict__ b2, const float* __restrict__ w3, const float* __restrict__ b3,
                                   int H, int A, float* __restrict__ w23, float* __restrict__ b23) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (H + 1) * A) return;
    const int k = i / A, a = i % A;
    const float* row = k < H ? w2 + (size_t)k * H : b2;
    double acc = k < H ? 0.0 : (double)b3[a];
    for (int j = 0; j < H; ++j) acc += (double)row[j] * (double)w3[(size_t)j * A + a];
    if (k < H) w23[(size_t)k * A + a] = (float)acc; else b23[a] = (float)acc;
}
// w0p[k][c]: k < A -> W_in[k], A <= k < A+Do -> W_in[k+td], else 0.   (skip = td for actor, 0 for critic with A=0)
__global__ void pack_w0_kernel(const float* __restrict__ win, int A, int skip, int Do, int KP, int H,
                               float* __restrict__ w0p) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= KP * H) return;
    int k = i / H, c = i % H;
    float v = 0.f;
    if (k < A) v = win[(size_t)k * H + c];
    else if (k < A + Do) v = win[(size_t)(k + skip) * H + c];
    w0p[i] = v;
}
// h0p[r][KP] = [x[r][0:A] | obs[rmap(r)][0:Do] | 0]; obs row = r / obs_div (get_logprobs tiles obs K times)
__global__ void pack_h0_kernel(const float* __restrict__ x, const float* __restrict__ obs, int N, int A, int Do,
                               int KP, int obs_div, float* __restrict__ h0p) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * KP) return;
    int r = (int)(i / KP), k = (int)(i % KP);
    float v = 0.f;
    if (k < A) v = x[(size_t)r * A + k];
    else if (k < A + Do) v = obs[(size_t)(r / obs_div) * Do + (k - A)];
    h0p[i] = v;
}
// trow[r] = mode 0: K-1 - inds[r];  mode 1: K-1 - (r % K)
__global__ void make_trow_kernel(const int* __restrict__ inds, int N, int K, int mode, int* __restrict__ trow) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= N) return;
    trow[r] = mode == 0 ? (K - 1 - inds[r]) : (K - 1 - (r % K));
}

// =====================================================================================
// Sampling epilogue (diffusion_vpg.py:198-206,239-243,301-338) for the layer-by-layer path
// =====================================================================================
struct SampleHyper {
    float dcv, rcv, facv, min_std; int deterministic;
};
// per-denoising-step constants (one gather per step instead of one per element)
struct StepConst { float sr, srm1, c1, c2, sd; };
__device__ __forceinline__ StepConst step_const(const float* __restrict__ sch, int T, int t) {
    StepConst c;
    c.sr = sch[SCH_SQRT_RECIP * T + t]; c.srm1 = sch[SCH_SQRT_RECIPM1 * T + t];
    c.c1 = sch[SCH_COEF1 * T + t]; c.c2 = sch[SCH_COEF2 * T + t];
    c.sd = expf(0.5f * sch[SCH_LOGVAR * T + t]);
    return c;
}
// sampling std of step t (diffusion_vpg.py:301-315)
__device__ __forceinline__ float sample_std(const StepConst& c, int t, const SampleHyper& hp) {
    if (hp.deterministic) return (t == 0) ? 0.f : fminf(fmaxf(c.sd, 1e-3f), 1e6f);
    return fminf(fmaxf(c.sd, hp.min_std), 1e6f);
}
__device__ __forceinline__ float ddpm_step_elem_c(float x, float eps, float noise, const StepConst& c, float sd, const SampleHyper& hp, bool last) {
    float xr = c.sr * x - c.srm1 * eps;
    if (hp.dcv >= 0.f) xr = fminf(fmaxf(xr, -hp.dcv), hp.dcv);
    float mu = c.c1 * xr + c.c2 * x;
    float nz = fminf(fmaxf(noise, -hp.rcv), hp.rcv);
    float xn = mu + sd * nz;
    if (last && hp.facv >= 0.f) xn = fminf(fmaxf(xn, -hp.facv), hp.facv);
    return xn;
}
__device__ __forceinline__ float ddpm_step_elem(float x, float eps, float noise, int t, const float* __restrict__ sch, int T,
                                                const SampleHyper hp, bool last) {
    const StepConst c = step_const(sch, T, t);
    return ddpm_step_elem_c(x, eps, noise, c, sample_std(c, t, hp), hp, last);
}
__global__ void sample_init_kernel(float* __restrict__ x, const float* __restrict__ xT, int B, int A,
                                   uint64_t seed, uint64_t offset, int64_t row_offset,
                                   float* __restrict__ chains, int K, int record) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * A) return;
    int r = i / A, a = i % A;
    float v = xT ? xT[i] : philox_normal(seed, offset, row_offset + r, 0, a);
    x[i] = v;
    if (record && chains) chains[((size_t)r * (K + 1)) * A + a] = v;
}
__global__ void sample_update_kernel(float* __restrict__ x, const float* __restrict__ eps, const float* __restrict__ noise,
                                     int B, int A, int t, int step, const float* __restrict__ sch, int T, SampleHyper hp,
                                     uint64_t seed, uint64_t offset, int64_t row_offset,
                                     float* __restrict__ chains, int K, int chain_slot, float* __restrict__ actions) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * A) return;
    int r = i / A, a = i % A;
    float nz = noise ? noise[(size_t)step * B * A + i] : philox_normal(seed, offset, row_offset + r, 1 + step, a);
    float xn = ddpm_step_elem(x[i], eps[i], nz, t, sch, T, hp, t == 0);
    x[i] = xn;
    if (chains && chain_slot >= 0) chains[((size_t)r * (K + 1) + chain_slot) * A + a] = xn;
    if (t == 0) actions[i] = xn;
}

// =====================================================================================
// Log-prob epilogue (diffusion_vpg.py:417-422, tfp Normal.log_prob)
// =====================================================================================
// Gaussian log-prob of one element given the step constants; sd already clipped, lgs = 0.5 log(2 pi) + log(sd)
__device__ __forceinline__ float logprob_elem_c(float x, float eps, float nxt, const StepConst& c, float sd, float lgs, float dcv,
                                                float* z_out, bool* inclip) {
    float xr = c.sr * x - c.srm1 * eps;
    bool in = true;
    if (dcv >= 0.f) { in = (xr >= -dcv && xr <= dcv); xr = fminf(fmaxf(xr, -dcv), dcv); }
    float mu = c.c1 * xr + c.c2 * x;
    float z = nxt / sd - mu / sd;
    if (z_out) { *z_out = z; *inclip = in; }
    return -0.5f * z * z - lgs;
}
__device__ __forceinline__ float logprob_std(const StepConst& c, float min_lp_std) { return fminf(fmaxf(c.sd, min_lp_std), 1e6f); }
__device__ __forceinline__ float logprob_elem(float x, float eps, float nxt, int t, const float* __restrict__ sch, int T,
                                              float dcv, float min_lp_std, float* z_out, float* sd_out, bool* inclip) {
    const StepConst c = step_const(sch, T, t);
    const float sd = logprob_std(c, min_lp_std);
    if (sd_out) *sd_out = sd;
    return logprob_elem_c(x, eps, nxt, c, sd, 0.91893853320467274f + logf(sd), dcv, z_out, inclip);
}
// prev/next either separate [N][A] arrays or derived from chains[B][K+1][A] with row = b*K+k
__global__ void logprob_kernel(const float* __restrict__ prev, const float* __restrict__ nxt, const float* __restrict__ chains,
                               const float* __restrict__ eps, const int* __restrict__ trow, int N, int A, int K,
                               const float* __restrict__ sch, int T, float dcv, float min_lp_std, float* __restrict__ logp) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * A) return;
    int r = (int)(i / A), a = (int)(i % A);
    float x, nx;
    if (chains) {
        int b = r / K, k = r % K;
        x = chains[((size_t)b * (K + 1) + k) * A + a];
        nx = chains[((size_t)b * (K + 1) + k + 1) * A + a];
    } else { x = prev[i]; nx = nxt[i]; }
    logp[i] = logprob_elem(x, eps[i], nx, trow[r], sch, T, dcv, min_lp_std, nullptr, nullptr, nullptr);
}
// gather prev rows from a chains tensor (for pack_h0 on get_logprobs)
__global__ void chains_prev_kernel(const float* __restrict__ chains, int N, int A, int K, float* __restrict__ prev) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * A) return;
    int r = (int)(i / A), a = (int)(i % A);
    int b = r / K, k = r % K;
    prev[i] = chains[((size_t)b * (K + 1) + k) * A + a];
}

// =====================================================================================
// PPO loss + gradient seed (diffusion_ppo.py:32-132).  One thread per row.
// sums[0..4] = sum pg, sum 0.5*(v-ret)^2 (or clipped variant), sum clipfrac, sum kl, sum ratio  (double partials per block)
// =====================================================================================
struct PpoHyper {
    int A, Da, K, T, reward_horizon, norm_adv;
    float dcv, min_lp_std, lp_lo, lp_hi, gamma_d, clip_coef, clip_base, clip_rate, clip_v, vf_coef;
    float inv_nglobal;
};
static PpoHyper ppo_hyper(const dppo_handle* h, int64_t N_global) {
    const dppo_cfg& c = h->cfg;
    PpoHyper hp;
    hp.A = h->g.A; hp.Da = c.action_dim; hp.K = h->g.K; hp.T = h->g.T; hp.reward_horizon = c.reward_horizon; hp.norm_adv = c.norm_adv;
    hp.dcv = c.denoised_clip_value; hp.min_lp_std = c.min_logprob_denoising_std;
    hp.lp_lo = c.logprob_clip_lo; hp.lp_hi = c.logprob_clip_hi; hp.gamma_d = c.gamma_denoising;
    hp.clip_coef = c.clip_ploss_coef; hp.clip_base = c.clip_ploss_coef_base; hp.clip_rate = c.clip_ploss_coef_rate;
    hp.clip_v = c.clip_vloss_coef; hp.vf_coef = c.vf_coef; hp.inv_nglobal = 1.0f / (float)N_global;
    return hp;
}
// The per-row loss math of every loss kernel (the kernels differ in row layout, loads, seed formula and reductions only).
// Policy part from the row's means of the clamped new / old log-probs, the raw advantage and the denoising index:
// dnew = d loss / d newm for this row, already scaled by 1 / N_global.
struct PpoRowPolicy { float pg, clipc, ratio, logratio, dnew; };
__device__ __forceinline__ PpoRowPolicy ppo_row_policy(float newm, float oldm, float adv, const float* __restrict__ advstats, int ind,
                                                       const PpoHyper& hp) {
    PpoRowPolicy o;
    if (hp.norm_adv) adv = (adv - advstats[0]) / (advstats[1] + 1e-8f);
    adv *= powf(hp.gamma_d, (float)(hp.K - ind - 1));
    o.logratio = newm - oldm; o.ratio = expf(o.logratio);
    // exponential clip schedule over the denoising index; K = 1 takes clip coefficient 0 (the reference divides 0 by 0)
    const float tt = hp.K > 1 ? (float)ind / (float)(hp.K - 1) : (float)ind;
    o.clipc = hp.K > 1 ? hp.clip_base + (hp.clip_coef - hp.clip_base) * (expf(hp.clip_rate * tt) - 1.f) / (expf(hp.clip_rate) - 1.f) : tt;
    const float rc = fminf(fmaxf(o.ratio, 1.f - o.clipc), 1.f + o.clipc);
    const float pg1 = -adv * o.ratio, pg2 = -adv * rc;
    o.pg = fmaxf(pg1, pg2);
    // d pg / d ratio: tf.maximum sends the gradient to pg1 on ties; clip_by_value passes inside the range
    const float dpg = (pg1 >= pg2) ? -adv : ((o.ratio >= 1.f - o.clipc && o.ratio <= 1.f + o.clipc) ? -adv : 0.f);
    o.dnew = dpg * o.ratio * hp.inv_nglobal;
    return o;
}
// value loss of the row (clipped when clip_v >= 0; *oldvalue is read only then) and its seed vf_coef * dv / N_global
struct PpoRowValue { float vl, seed; };
__device__ __forceinline__ PpoRowValue ppo_row_value(float v, float ret, const float* __restrict__ oldvalue, const PpoHyper& hp) {
    float vl, dv;
    if (hp.clip_v >= 0.f) {
        const float ov = *oldvalue;
        const float un = (v - ret) * (v - ret);
        const float dcl = v - ov;
        const float vc = ov + fminf(fmaxf(dcl, -hp.clip_v), hp.clip_v);
        const float cl = (vc - ret) * (vc - ret);
        if (un >= cl) { vl = 0.5f * un; dv = (v - ret); }
        else { vl = 0.5f * cl; dv = (dcl >= -hp.clip_v && dcl <= hp.clip_v) ? (vc - ret) : 0.f; }
    } else { vl = 0.5f * (v - ret) * (v - ret); dv = (v - ret); }
    return {vl, hp.vf_coef * dv * hp.inv_nglobal};
}
// the row's terms of the five metric sums
__device__ __forceinline__ void ppo_row_metrics(double acc[5], const PpoRowPolicy& p, float vl) {
    acc[0] = p.pg; acc[1] = vl; acc[2] = (fabsf(p.ratio - 1.f) > p.clipc) ? 1.0 : 0.0;
    acc[3] = (p.ratio - 1.f) - p.logratio; acc[4] = p.ratio;
}
// flat != nullptr: row i of the minibatch is rollout row flat[i] / K (index-driven minibatch); out-of-range indices read row 0
__global__ void adv_stats_kernel(const float* __restrict__ adv, int N, float* __restrict__ out /*mean,std*/,
                                 const int* __restrict__ flat = nullptr, int K = 1, long long P = 0) {
    __shared__ double s1[1024], s2[1024];
    double a = 0, b = 0;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        size_t src = i;
        if (flat) { const int f = flat[i]; src = (f < 0 || (long long)f >= P * K) ? 0 : (size_t)(f / K); }
        double v = adv[src]; a += v; b += v * v;
    }
    s1[threadIdx.x] = a; s2[threadIdx.x] = b;
    __syncthreads();
    for (int o = blockDim.x >> 1; o > 0; o >>= 1) {
        if (threadIdx.x < o) { s1[threadIdx.x] += s1[threadIdx.x + o]; s2[threadIdx.x] += s2[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        double mean = s1[0] / N, var = s2[0] / N - mean * mean;
        out[0] = (float)mean; out[1] = (float)sqrt(var > 0 ? var : 0);
    }
}
__global__ void set_scalars_kernel(float* dst, float a, float b) { dst[0] = a; dst[1] = b; }

__global__ void __launch_bounds__(128) ppo_loss_kernel(
    const float* __restrict__ prev, const float* __restrict__ nxt, const float* __restrict__ eps,
    const int* __restrict__ inds, const float* __restrict__ returns, const float* __restrict__ oldvalues,
    const float* __restrict__ advantages, const float* __restrict__ oldlogp, const float* __restrict__ newvalues,
    const float* __restrict__ advstats, const float* __restrict__ sch, PpoHyper hp, int N,
    float* __restrict__ deps, float* __restrict__ dvalue, double* __restrict__ block_sums) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    double acc[5] = {0, 0, 0, 0, 0};
    if (r < N) {
        const int A = hp.A, ind = inds[r], t = hp.K - 1 - ind;
        const int nuse = min(hp.reward_horizon, A / hp.Da) * hp.Da;   // newlogprobs[:, :reward_horizon, :]
        float newm = 0.f, oldm = 0.f;
        for (int a = 0; a < nuse; ++a) {
            size_t i = (size_t)r * A + a;
            float lp = logprob_elem(prev[i], eps[i], nxt[i], t, sch, hp.T, hp.dcv, hp.min_lp_std, nullptr, nullptr, nullptr);
            newm += fminf(fmaxf(lp, hp.lp_lo), hp.lp_hi);
            oldm += fminf(fmaxf(oldlogp[i], hp.lp_lo), hp.lp_hi);
        }
        newm /= (float)nuse; oldm /= (float)nuse;
        const PpoRowPolicy p = ppo_row_policy(newm, oldm, advantages[r], advstats, ind, hp);
        for (int a = 0; a < A; ++a) {
            size_t i = (size_t)r * A + a;
            float g = 0.f;
            if (a < nuse) {
                float z, sd; bool in;
                float lp = logprob_elem(prev[i], eps[i], nxt[i], t, sch, hp.T, hp.dcv, hp.min_lp_std, &z, &sd, &in);
                if (lp >= hp.lp_lo && lp <= hp.lp_hi && in)
                    g = p.dnew / (float)nuse * (z / sd) * sch[SCH_COEF1 * hp.T + t] * (-sch[SCH_SQRT_RECIPM1 * hp.T + t]);
            }
            deps[i] = g;
        }
        const PpoRowValue vr = ppo_row_value(newvalues[r], returns[r], oldvalues + r, hp);
        dvalue[r] = vr.seed;
        ppo_row_metrics(acc, p, vr.vl);
    }
    __shared__ double red[5][128];
    for (int k = 0; k < 5; ++k) red[k][threadIdx.x] = acc[k];
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if (threadIdx.x < o) for (int k = 0; k < 5; ++k) red[k][threadIdx.x] += red[k][threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x < 5) block_sums[(size_t)blockIdx.x * 5 + threadIdx.x] = red[threadIdx.x][0];
}
// sums the per-block partials; writes metric partial sums (already divided by N_global) to dst[0..7]
// body shared by ppo_metrics_kernel and the merged tail kernel: threads >= 256 of a larger block only take part in the barriers
__device__ __forceinline__ void ppo_metrics_body(const double* __restrict__ block_sums, int nblocks, float inv_nglobal, float frac_local,
                                                 float* __restrict__ dst) {
    __shared__ double red[5][256];
    const int tid = threadIdx.x;
    double a[5] = {0, 0, 0, 0, 0};
    if (tid < 256) {
        for (int b = tid; b < nblocks; b += 256)
            for (int k = 0; k < 5; ++k) a[k] += block_sums[(size_t)b * 5 + k];
        for (int k = 0; k < 5; ++k) red[k][tid] = a[k];
    }
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o) for (int k = 0; k < 5; ++k) red[k][tid] += red[k][tid + o];
        __syncthreads();
    }
    if (tid == 0) {
        dst[0] = (float)(red[0][0] * inv_nglobal);   // pg_loss
        dst[1] = -frac_local;                         // entropy_loss = -mean(eta) = -1 (eta == 1 for DDPM)
        dst[2] = (float)(red[1][0] * inv_nglobal);   // v_loss
        dst[3] = (float)(red[2][0] * inv_nglobal);   // clipfrac
        dst[4] = (float)(red[3][0] * inv_nglobal);   // approx_kl
        dst[5] = (float)(red[4][0] * inv_nglobal);   // mean ratio
        dst[6] = 0.f;                                 // bc_loss
        dst[7] = frac_local;                          // mean eta
    }
}
__global__ void ppo_metrics_kernel(const double* __restrict__ block_sums, int nblocks, float inv_nglobal, float frac_local,
                                   float* __restrict__ dst) {
    ppo_metrics_body(block_sums, nblocks, inv_nglobal, frac_local, dst);
}

// minibatch assembly from the resident rollout buffers (train_ppo_diffusion_agent.py:293-312): one thread per output float
__global__ void gather_minibatch_kernel(const float* __restrict__ obs_buf, const float* __restrict__ chains_buf, const float* __restrict__ oldlogp_buf,
                                        const float* __restrict__ ret_buf, const float* __restrict__ val_buf, const float* __restrict__ adv_buf,
                                        const int* __restrict__ inds_k, int N, int K, int A, int Do, long long P,
                                        float* __restrict__ obs, float* __restrict__ prev, float* __restrict__ nxt, float* __restrict__ olp,
                                        int* __restrict__ dind, float* __restrict__ ret, float* __restrict__ val, float* __restrict__ adv, int* __restrict__ bad) {
    const int W = Do + 3 * A + 4;                      // floats produced per row
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * W) return;
    const int r = (int)(i / W), c = (int)(i % W);
    const int flat = inds_k[r];
    if (flat < 0 || (long long)flat >= P * K) { if (c == 0) atomicOr(bad, 1); return; }
    const size_t b = (size_t)(flat / K); const int k = flat % K;
    if (c < Do) obs[(size_t)r * Do + c] = obs_buf[b * Do + c];
    else if (c < Do + A) prev[(size_t)r * A + (c - Do)] = chains_buf[(b * (K + 1) + k) * A + (c - Do)];
    else if (c < Do + 2 * A) nxt[(size_t)r * A + (c - Do - A)] = chains_buf[(b * (K + 1) + k + 1) * A + (c - Do - A)];
    else if (c < Do + 3 * A) olp[(size_t)r * A + (c - Do - 2 * A)] = oldlogp_buf[(b * K + k) * A + (c - Do - 2 * A)];
    else if (c == Do + 3 * A) dind[r] = k;
    else if (c == Do + 3 * A + 1) ret[r] = ret_buf[b];
    else if (c == Do + 3 * A + 2) val[r] = val_buf[b];
    else adv[r] = adv_buf[b];
}

// GAE backward scan, one thread per env (train_ppo_diffusion_agent.py:242-263).  Explicit round-to-nearest double
// multiplies / adds in NumPy's evaluation order (no FMA contraction), so the result is bit-identical to the reference.
__global__ void gae_kernel(const double* __restrict__ rewards, const float* __restrict__ terminated, const float* __restrict__ values,
                           const float* __restrict__ next_values, int S, int E, double rsc, double gamma, double lam,
                           float* __restrict__ adv, float* __restrict__ ret) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    double last = 0.0;
    for (int t = S - 1; t >= 0; --t) {
        const size_t i = (size_t)t * E + e;
        // gamma * nextvalues: at the last step nextvalues is the critic's fp32 output and NumPy multiplies a Python float into an fp32
        // array IN fp32 (train_ppo_diffusion_agent.py:252,259); earlier steps read the float64 values_trajs holder
        const double gnext = (t == S - 1) ? (double)__fmul_rn((float)gamma, next_values[e]) : __dmul_rn(gamma, (double)values[i + E]);
        const double nonterm = 1.0 - (double)terminated[i];
        const double v = (double)values[i];
        // delta = r * rsc + gamma * nextv * nonterm - v
        const double delta = __dsub_rn(__dadd_rn(__dmul_rn(rewards[i], rsc), __dmul_rn(gnext, nonterm)), v);
        // last = delta + gamma * lam * nonterm * last
        last = __dadd_rn(delta, __dmul_rn(__dmul_rn(__dmul_rn(gamma, lam), nonterm), last));
        adv[i] = (float)last;
        ret[i] = (float)__dadd_rn(last, v);
    }
}

// pre-train: x_noisy = sqrt(acp_t) x0 + sqrt(1-acp_t) noise (diffusion.py:196-202); also materialises t / noise draws
__global__ void pretrain_prep_kernel(const float* __restrict__ x0, const int* __restrict__ t_in, const float* __restrict__ noise_in,
                                     int N, int A, int T, const float* __restrict__ sch, uint64_t seed, uint64_t offset,
                                     int64_t row_offset, int* __restrict__ trow, float* __restrict__ noise, float* __restrict__ xn) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * A) return;
    int r = (int)(i / A), a = (int)(i % A);
    int t = t_in ? t_in[r] : (int)(((uint64_t)philox_uint(seed, offset, row_offset + r, 255) * (uint64_t)T) >> 32);
    float nz = noise_in ? noise_in[i] : philox_normal(seed, offset, row_offset + r, 0, a);
    if (a == 0) trow[r] = t;
    noise[i] = nz;
    xn[i] = sch[SCH_SQRT_ACP * T + t] * x0[i] + sch[SCH_SQRT_1M_ACP * T + t] * nz;
}
// loss = mean((eps - noise)^2); deps = 2 (eps - noise) / (N_global * A)
__global__ void __launch_bounds__(256) mse_loss_kernel(const float* __restrict__ eps, const float* __restrict__ noise, size_t n,
                                                       float scale, float* __restrict__ deps, double* __restrict__ block_sums) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    double a = 0;
    if (i < n) { float d = eps[i] - noise[i]; deps[i] = 2.f * d * scale; a = (double)d * d; }
    __shared__ double red[256];
    red[threadIdx.x] = a;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) block_sums[blockIdx.x] = red[0];
}
__global__ void sum_blocks_kernel(const double* __restrict__ block_sums, int nblocks, float scale, float* __restrict__ dst) {
    __shared__ double red[256];
    double a = 0;
    for (int b = threadIdx.x; b < nblocks; b += blockDim.x) a += block_sums[b];
    red[threadIdx.x] = a;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) dst[0] = (float)(red[0] * scale);
}

// =====================================================================================
// Column sums (bias gradients) and per-t column sums (time-embedding gradient)
//   part[blk][seg][n] = sum over this block's rows with seg(row)==seg of D[row][n]
// Block (x, y) takes row block x and the columns [y * slice, (y + 1) * slice) of every segment (shared memory [nseg][slice]).
// =====================================================================================
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ D, int ld, int N, int ncols, int slice,
                                                     const int* __restrict__ seg, int nseg, int rows_per_block,
                                                     float* __restrict__ part) {
    extern __shared__ float sm[];   // [nseg][slice]
    const int c0 = blockIdx.y * slice, nc = min(slice, ncols - c0);
    for (int i = threadIdx.x; i < nseg * slice; i += blockDim.x) sm[i] = 0.f;
    __syncthreads();
    const int r0 = blockIdx.x * rows_per_block, r1 = min(N, r0 + rows_per_block);
    // each thread owns columns c = tid, tid+256, ... of the slice and walks the rows: no atomics needed
    for (int c = threadIdx.x; c < nc; c += blockDim.x) {
        for (int r = r0; r < r1; ++r) {
            int s = seg ? seg[r] : 0;
            sm[s * slice + c] += D[(size_t)r * ld + c0 + c];
        }
    }
    __syncthreads();
    float* out = part + (size_t)blockIdx.x * nseg * ncols + c0;
    for (int i = threadIdx.x; i < nseg * nc; i += blockDim.x) out[(size_t)(i / nc) * ncols + i % nc] = sm[(i / nc) * slice + i % nc];
}

// time-MLP + layer-0 bias backward from G[T][H] = per-t column sums of du, on time_backward_grid() blocks of 512 threads
// (`bid` of a stand-alone launch or of a block range of the merged tail kernel):
//  * blocks [0, T): dte[t][j] = sum_c W_in[A+j][c] G[t][c] for t = bid, one warp per j (lane-strided columns, butterfly), into
//    dte_g [T][td]; the LAST of these blocks to finish (counter dte_g[T*td], left at zero) runs the time MLP's backward from the
//    T rows: dh, dW2 / dW1 of the time MLP and their biases, every operand in shared memory (the T-long loops of a single block
//    walking L2 were the whole cost of the first version: ~58 k cycles);
//  * blocks [T, ..): db_in and the td time rows of dW_in for 32 columns each, 16 threads per column over j.
// Every output keeps the summation order of the single-block version (t ascending; c ascending per lane, then the butterfly).
__device__ __forceinline__ void time_backward_body(const int bid, float* sm,
                                     const float* __restrict__ w, ActorOff o, int A, int td, int H, int T,
                                     const float* __restrict__ G, const float* __restrict__ sinemb,
                                     const float* __restrict__ thpre, const float* __restrict__ temb,
                                     float* __restrict__ dte_g, float* __restrict__ g) {
    const int tid = threadIdx.x, nt = blockDim.x;
    if (bid >= T) {
        const int lanes = 16;                           // threads per column
        const int c0 = (bid - T) * (nt / lanes), c1 = min(H, c0 + nt / lanes);
        for (int i = tid; i < (c1 - c0) * lanes; i += nt) {
            const int c = c0 + i / lanes, part = i % lanes;
            // the T values of column c are loaded up front (independent loads: one L2 latency instead of T)
            float bsum = 0.f;
            float acc[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) acc[q] = 0.f;
            for (int t0 = 0; t0 < T; t0 += 32) {
                float gc[32];
#pragma unroll
                for (int q = 0; q < 32; ++q) gc[q] = (t0 + q < T) ? G[(size_t)(t0 + q) * H + c] : 0.f;
#pragma unroll
                for (int q = 0; q < 32; ++q) bsum += gc[q];
#pragma unroll
                for (int jj = 0; jj < 2; ++jj) {
                    const int j = part + jj * lanes;
                    if (j < td) {
#pragma unroll
                        for (int q = 0; q < 32; ++q) if (t0 + q < T) acc[jj] = fmaf(temb[(t0 + q) * td + j], gc[q], acc[jj]);
                    }
                }
            }
            if (part == 0) g[o.bin + c] = bsum;
            for (int jj = 0; jj < 2; ++jj) {
                const int j = part + jj * lanes;
                if (j < td) g[o.win + (size_t)(A + j) * H + c] = acc[jj];
            }
            // time_dim > 2 * lanes: plain loop for the rest
            for (int j = part + 2 * lanes; j < td; j += lanes) {
                float a = 0.f;
                for (int t = 0; t < T; ++t) a = fmaf(temb[t * td + j], G[(size_t)t * H + c], a);
                g[o.win + (size_t)(A + j) * H + c] = a;
            }
        }
        return;
    }
    // d temb[t][j]: a warp walks its W_in row and the G row (H <= 1024)
    {
        const int t = bid, lane = tid & 31;
        for (int j = tid >> 5; j < td; j += nt >> 5) {
            float s = 0.f;
#pragma unroll
            for (int q0 = 0; q0 < 32; q0 += 16) {       // 16 columns of both rows in flight at once
                float wr[16], gv[16];
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const int c = lane + (q0 + q) * 32;
                    wr[q] = c < H ? w[o.win + (size_t)(A + j) * H + c] : 0.f;
                    gv[q] = c < H ? G[(size_t)t * H + c] : 0.f;
                }
#pragma unroll
                for (int q = 0; q < 16; ++q) { const int c = lane + (q0 + q) * 32; if (c < H) s = fmaf(wr[q], gv[q], s); }
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
            if (lane == 0) dte_g[t * td + j] = s;
        }
    }
    __shared__ int last_flag;
    int* done = reinterpret_cast<int*>(dte_g + T * td);
    __threadfence();
    __syncthreads();
    if (tid == 0) last_flag = (atomicAdd(done, 1) == T - 1) ? 1 : 0;
    __syncthreads();
    if (!last_flag) return;
    __threadfence();
    float* dte = sm;                 // [T][td]
    float* dh = dte + T * td;        // [T][2td]
    float* mt = dh + T * 2 * td;     // [T][2td] mish(thpre)
    for (int i = tid; i < T * td; i += nt) dte[i] = __ldcg(dte_g + i);
    for (int i = tid; i < T * 2 * td; i += nt) mt[i] = mish_f(thpre[i]);
    __syncthreads();
    for (int i = tid; i < T * 2 * td; i += nt) {    // d hidden pre-activation
        int t = i / (2 * td), k = i % (2 * td);
        float s = 0.f;
        for (int j = 0; j < td; ++j) s = fmaf(w[o.tw2 + (size_t)k * td + j], dte[t * td + j], s);
        dh[i] = s * mish_grad_f(thpre[i]);
    }
    __syncthreads();
    for (int i = tid; i < 2 * td * td; i += nt) {   // dW2[k][j], dW1[s][k]
        int k = i / td, j = i % td;
        float s = 0.f;
        for (int t = 0; t < T; ++t) s = fmaf(mt[t * 2 * td + k], dte[t * td + j], s);
        g[o.tw2 + i] = s;
        int ss = i / (2 * td), kk = i % (2 * td);
        float a = 0.f;
        for (int t = 0; t < T; ++t) a = fmaf(sinemb[t * td + ss], dh[t * 2 * td + kk], a);
        g[o.tw1 + i] = a;
    }
    for (int j = tid; j < td; j += nt) { float s = 0.f; for (int t = 0; t < T; ++t) s += dte[t * td + j]; g[o.tb2 + j] = s; }
    for (int k = tid; k < 2 * td; k += nt) { float s = 0.f; for (int t = 0; t < T; ++t) s += dh[t * 2 * td + k]; g[o.tb1 + k] = s; }
    if (tid == 0) *done = 0;                         // ready for the next launch
}
__global__ void __launch_bounds__(512) time_backward_kernel(const float* __restrict__ w, ActorOff o, int A, int td, int H, int T,
                                     const float* __restrict__ G, const float* __restrict__ sinemb,
                                     const float* __restrict__ thpre, const float* __restrict__ temb,
                                     float* __restrict__ dte_g, float* __restrict__ g) {
    extern __shared__ float sm[];
    time_backward_body(blockIdx.x, sm, w, o, A, td, H, T, G, sinemb, thpre, temb, dte_g, g);
}
static inline int time_backward_grid(const Geom& g) { return g.T + (g.H + 31) / 32; }
static inline size_t time_backward_smem(const Geom& g) { return (size_t)5 * g.T * g.td * sizeof(float); }
// the time-MLP / layer-0 bias backward of actor `net` from G [T][H] into its gradient slice gnet
static cudaError_t launch_time_backward(const dppo_handle* h, cudaStream_t s, int net, const float* G, float* gnet) {
    // the attribute is per device and shared by every handle on it: raised whenever a handle needs more than is set
    static size_t attr_dev[64] = {};
    const Geom& g = h->g; const ActorDerived& d = h->ad[net];
    const size_t sm = time_backward_smem(g);
    if (sm > 48 * 1024 && sm > attr_dev[h->device & 63]) {
        const cudaError_t e = cudaFuncSetAttribute(time_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        if (e != cudaSuccess) return e;
        attr_dev[h->device & 63] = sm;
    }
    time_backward_kernel<<<time_backward_grid(g), 512, sm, s>>>(h->net_w[net], g.ao, g.A, g.td, g.H, g.T, G, d.sinemb, d.thpre, d.temb, d.dte, gnet);
    return cudaGetLastError();
}
// scatter dW0p[KP][H] rows back into dW_in: k < A -> row k; A <= k < A+Do -> row k+skip
__device__ __forceinline__ void unpack_dw0_body(const int bid, const float* __restrict__ dw0p, int A, int skip, int Do, int H, float* __restrict__ gwin) {
    int i = bid * blockDim.x + threadIdx.x;
    if (i >= (A + Do) * H) return;
    int k = i / H, c = i % H;
    gwin[(size_t)(k < A ? k : k + skip) * H + c] = dw0p[i];
}
__global__ void unpack_dw0_kernel(const float* __restrict__ dw0p, int A, int skip, int Do, int H, float* __restrict__ gwin) {
    unpack_dw0_body(blockIdx.x, dw0p, A, skip, Do, H, gwin);
}

// =====================================================================================
// Keras-3 AdamW (decoupled decay first, then Adam with folded bias correction)
// =====================================================================================
// one element: every kernel that applies the update calls this, so that the arithmetic (and its contraction) cannot differ
__device__ __forceinline__ void adamw_elem(float& p, float& mi, float& vi, float gi, float lr, float alpha, float b1, float b2, float eps, float wd) {
    if (wd != 0.f) p = p - p * (wd * lr);
    mi = mi + (gi - mi) * (1.f - b1);
    vi = vi + (gi * gi - vi) * (1.f - b2);
    p = p - mi * alpha / (sqrtf(vi) + eps);
}
// skip[0] | skip[1] != 0 (optional device flags: bad minibatch indices, a peer barrier that timed out): leave everything untouched
__global__ void adamw_kernel(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                             size_t n, float lr, float alpha, float b1, float b2, float eps, float wd,
                             const int* __restrict__ skip0 = nullptr, const int* __restrict__ skip1 = nullptr) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if ((skip0 && *skip0) || (skip1 && *skip1)) return;
    float p = w[i], mi = m[i], vi = v[i];
    adamw_elem(p, mi, vi, g[i], lr, alpha, b1, b2, eps, wd);
    w[i] = p; m[i] = mi; v[i] = vi;
}
// tf.clip_by_norm on every variable of the flat gradient (train_ppo_diffusion_agent.py:352): one block per variable,
// g <- g * c / max(||g||_2, c)   (l2sum == 0 -> norm 1, like TF's guarded sqrt)
struct VarSegs { unsigned int off[24]; int n; };
__global__ void __launch_bounds__(1024) clip_by_norm_kernel(float* __restrict__ g, VarSegs segs, float clip) {
    const unsigned int b = segs.off[blockIdx.x], e = segs.off[blockIdx.x + 1];
    float acc = 0.f;
    for (unsigned int i = b + threadIdx.x; i < e; i += blockDim.x) { const float x = g[i]; acc = fmaf(x, x, acc); }
    __shared__ float part[32];
    __shared__ float denom;
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        float t = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.f;
        for (int o = 16; o; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (threadIdx.x == 0) denom = fmaxf(sqrtf(t > 0.f ? t : 1.f), clip);
    }
    __syncthreads();
    const float d = denom;
    if (d == clip) return;                                   // norm <= clip: g * c / c
    for (unsigned int i = b + threadIdx.x; i < e; i += blockDim.x) g[i] = g[i] * clip / d;
}
// ---- peer-memory gradient all-reduce fused with AdamW (one node, P2P over NVLink / NVSwitch)
struct PeerPtrs { const float* g[8]; unsigned long long* flags[8]; };
// flag barrier: tell every peer "my gradient buffer of this epoch is complete", wait until all peers said so
// A rank may arrive long before its peers (each steps its own host envs): the wait is bounded by `timeout_cycles` (host: seconds x
// SM clock, DPPO_PEER_TIMEOUT_S, default 600 s) and a timeout does NOT trap - it raises status[0], which makes the reduce / AdamW
// kernels that follow no-ops (weights and optimizer state stay intact) and is reported by the next host-side status check.
__global__ void peer_barrier_kernel(PeerPtrs pp, unsigned long long* my_flags, int rank, int world, unsigned long long epoch,
                                    long long timeout_cycles, int* __restrict__ status) {
    const int p = threadIdx.x;
    if (p >= world) return;
    if (*((volatile int*)status)) return;                       // an earlier barrier already failed
    __threadfence_system();
    *((volatile unsigned long long*)(pp.flags[p] + rank)) = epoch;
    const long long t0 = clock64();
    while (*((volatile unsigned long long*)(my_flags + p)) < epoch) {
        if (clock64() - t0 > timeout_cycles) {
            printf("peer barrier timed out: rank %d waiting for rank %d (epoch %llu)\n", rank, p, epoch);
            atomicExch(status, 1);
            break;
        }
        __nanosleep(64);
    }
    __threadfence_system();
}
// g_sum = sum over ranks (fixed order) of their gradient buffers; AdamW on the first n_param entries; the reduced vector
// (gradients ++ metric partial sums) is written back to this rank's buffer
__global__ void __launch_bounds__(256) peer_allreduce_adamw_kernel(PeerPtrs pp, int world, float* __restrict__ g_sum, float* __restrict__ w,
                                                                  float* __restrict__ m, float* __restrict__ v, size_t n_param, size_t n_total,
                                                                  float lr, float alpha, float b1, float b2, float eps, float wd,
                                                                  const int* __restrict__ skip0 = nullptr, const int* __restrict__ skip1 = nullptr) {
    const bool no_update = (skip0 && *skip0) || (skip1 && *skip1);
    if (skip1 && *skip1) return;                                   // failed barrier: the peers' buffers are not ready
    const size_t n4 = n_total / 4;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4 + (n_total & 3); i += (size_t)gridDim.x * blockDim.x) {
        float s[4] = {0.f, 0.f, 0.f, 0.f};
        const bool vec = i < n4;
        const size_t e0 = vec ? i * 4 : n4 * 4 + (i - n4);
        const int cnt = vec ? 4 : 1;
        for (int p = 0; p < world; ++p) {
            if (vec) { const float4 x = __ldcv(reinterpret_cast<const float4*>(pp.g[p]) + i); s[0] += x.x; s[1] += x.y; s[2] += x.z; s[3] += x.w; }
            else s[0] += __ldcv(pp.g[p] + e0);
        }
        for (int k = 0; k < cnt; ++k) {
            const size_t e = e0 + k;
            if (e < n_param && !no_update) {
                float pw = w[e], mi = m[e], vi = v[e]; const float gi = s[k];
                if (wd != 0.f) pw = pw - pw * (wd * lr);
                mi = mi + (gi - mi) * (1.f - b1);
                vi = vi + (gi * gi - vi) * (1.f - b2);
                pw = pw - mi * alpha / (sqrtf(vi) + eps);
                w[e] = pw; m[e] = mi; v[e] = vi;
            }
        }
        // this rank's gradient buffer is one of the summands its peers are still reading: the sum goes to a separate buffer
        if (vec) reinterpret_cast<float4*>(g_sum)[i] = make_float4(s[0], s[1], s[2], s[3]); else g_sum[e0] = s[0];
    }
}
// Two-shot variant for larger worlds: after the first flag barrier rank r sums ONLY its 1/world slice of every rank's gradient
// buffer (fixed order) and stores the result into the sum buffer of every rank (world-1 remote stores); a second flag barrier,
// then plain AdamW on the local copy of the sum.  Per rank n floats are read and n written over NVLink instead of world * n read.
struct PeerSums { float* s[8]; };
__global__ void __launch_bounds__(256) peer_reduce_scatter_bcast_kernel(PeerPtrs pp, PeerSums ps, int rank, int world, size_t n4, const int* __restrict__ status) {
    if (*status) return;
    const size_t per = (n4 + (size_t)world - 1) / (size_t)world, lo = (size_t)rank * per, hi = lo + per < n4 ? lo + per : n4;
    for (size_t i = lo + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (size_t)gridDim.x * blockDim.x) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int p = 0; p < world; ++p) { const float4 x = __ldcv(reinterpret_cast<const float4*>(pp.g[p]) + i); a.x += x.x; a.y += x.y; a.z += x.z; a.w += x.w; }
        for (int q = 0; q < world; ++q) reinterpret_cast<float4*>(ps.s[q])[i] = a;
    }
}
// metrics of an update whose minibatch indices were out of range (the AdamW step was skipped): NaN, so that a device-side caller cannot miss it
__global__ void poison_metrics_kernel(float* __restrict__ metrics8, const int* __restrict__ bad) {
    if (*bad && threadIdx.x < 8) metrics8[threadIdx.x] = __int_as_float(0x7fc00000);
}
__global__ void ema_kernel(float* __restrict__ ema, const float* __restrict__ w, size_t n, float decay) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) ema[i] = ema[i] * decay + w[i] * (1.f - decay);
}
