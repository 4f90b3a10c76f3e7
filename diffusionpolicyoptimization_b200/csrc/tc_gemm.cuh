// tcgen05 GEMM for sm_100a:  D[M,N] (+)= A[M,K] * B[K,N],  bf16 operands, fp32 accumulation in TMEM.
//
//   * operands are staged by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle) into a 4-stage
//     shared-memory ring; one elected thread issues tcgen05.mma (UMMA 128 x BN x 16);
//     accumulators live in TMEM (2 stages x BN columns) and are drained by 4 epilogue warps with
//     tcgen05.ld while the next tile's MMAs run (persistent CTAs, static tile round-robin).
//   * each operand is either K-major (the reduction index is contiguous in memory: activations
//     [rows][features] as A of a forward layer, W[in][out] as B of dX = dY W^T) or MN-major (the
//     M/N index is contiguous: W[in][out] as B of a forward layer, activations as BOTH operands of
//     dW = X^T dY) - so no tensor is ever transposed in memory.
//   * A may be the K-concatenation of two tensors ([a2 | h0]): the residual  u = h0 W_in  is folded
//     into the second layer's accumulation instead of being stored and re-read.
//   * fused epilogue: + bias, activation, * act'(mask), + residual, fp32 / bf16 (pre- and post-
//     activation) stores, split-K partial outputs.
#pragma once
#include <unordered_map>
#include "common.cuh"
#include <cuda.h>

namespace tc {

constexpr int BM = 128, BK = 64, STAGES = 4;
constexpr int NUM_THREADS = 192;      // warp 0: TMA, warp 1: MMA + TMEM alloc, warps 2..5: epilogue

struct Epi {
    int M, N;                         // valid extents of the output
    const float* bias;                // [N]
    int act;                          // 0 none, 1 relu, 2 mish
    const __nv_bfloat16* mask; int ldmask; int mask_mode;   // 1: *= (mask > 0), 2: *= mish'(mask)
    const __nv_bfloat16* add; int ldadd;                    // += add[m][n]
    float* out_f32; int ld_f32; size_t split_stride;        // fp32 row-major (+ split * split_stride)
    int f32_atomic;                                         // accumulate into out_f32 with red.global.add (split-K without partials)
    __nv_bfloat16* out_bf16; int ld_bf16;                   // bf16 row-major, post-activation
    __nv_bfloat16* out_pre; int ld_pre;                     // bf16 row-major, pre-activation
};

struct Params {
    int m_blocks, n_blocks, splits;
    int kblocks, kb_per_split;        // K blocks (of 64) in total / per split
    int ka_blocks;                    // K blocks taken from tensor map A (the rest from A2)
    Epi epi;
};

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait: a descriptor / byte-count bug must trap, never hang the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) { printf("tc_gemm: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x); __trap(); }
    }
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// one lane of a converged warp: keeps the issue warps' control flow warp-uniform so that nvcc emits the
// uniform-datapath instructions (UTCHMMA / UTCBAR / UTMALDG) without ELECT / BRA.U.ANY waterfall loops
__device__ __forceinline__ bool elect_one_lane() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P1;\n\telect.sync _|P1, 0xFFFFFFFF;\n\tselp.b32 %0, 1, 0, P1;\n\t}" : "=r"(pred));
    return pred != 0;
}
// shared-memory matrix descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor), 128B swizzle
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;          // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;          // SWIZZLE_128B
    return d;
}
__host__ __device__ constexpr uint32_t make_idesc(int umma_m, int umma_n, bool a_mn, bool b_mn, bool a_bf16 = true, bool b_bf16 = true) {
    return (1u << 4)                      // D format  : F32
         | ((a_bf16 ? 1u : 0u) << 7) | ((b_bf16 ? 1u : 0u) << 10)   // A, B format: BF16 (1) or F16 (0), chosen per operand
         | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16)
         | ((uint32_t)(umma_n >> 3) << 17) | ((uint32_t)(umma_m >> 4) << 24);
}

template <int BN> constexpr size_t smem_bytes() {
    return (size_t)STAGES * (BM * BK * 2 + BN * BK * 2) + 1024 /*align*/ + 256 /*barriers*/;
}

// =====================================================================================
template <int BN, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2,
            const __grid_constant__ CUtensorMap tmB, const Params p) {
    constexpr int A_STAGE = BM * BK * 2, B_STAGE = BN * BK * 2;
    constexpr int TMEM_COLS = (2 * BN <= 32) ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* sA = smem;
    uint8_t* sB = smem + STAGES * A_STAGE;
    uint64_t* bars = (uint64_t*)(smem + STAGES * (A_STAGE + B_STAGE));
    uint64_t* full = bars;                 // [STAGES]  TMA -> MMA
    uint64_t* empty = bars + STAGES;       // [STAGES]  MMA -> TMA
    uint64_t* tfull = bars + 2 * STAGES;   // [2]       MMA -> epilogue
    uint64_t* tempty = tfull + 2;          // [2]       epilogue -> MMA
    uint32_t* tmem_slot = (uint32_t*)(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles = p.m_blocks * p.n_blocks * p.splits;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmA2); tma_prefetch_desc(&tmB);
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    if (warp == 0) {
        // ===================== TMA producer (warp-uniform; an elected lane issues) =====================
        {
            int stage = 0; uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
                const int split = tile / (p.m_blocks * p.n_blocks);
                const int rem = tile % (p.m_blocks * p.n_blocks);
                const int m_blk = rem / p.n_blocks, n_blk = rem % p.n_blocks;
                const int kb0 = split * p.kb_per_split, kb1 = min(p.kblocks, kb0 + p.kb_per_split);
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    if (elect_one_lane()) {
                        mbar_expect_tx(&full[stage], A_STAGE + B_STAGE);
                        uint8_t* a = sA + stage * A_STAGE;
                        uint8_t* b = sB + stage * B_STAGE;
                        const CUtensorMap* ma = kb < p.ka_blocks ? &tmA : &tmA2;
                        const int ka = (kb < p.ka_blocks ? kb : kb - p.ka_blocks) * BK;
                        if (!A_MN) tma_load_2d(a, ma, &full[stage], ka, m_blk * BM);
                        else {
#pragma unroll
                            for (int j = 0; j < BM / 64; ++j) tma_load_2d(a + j * (64 * BK * 2), ma, &full[stage], m_blk * BM + j * 64, ka);
                        }
                        if (!B_MN) tma_load_2d(b, &tmB, &full[stage], kb * BK, n_blk * BN);
                        else {
#pragma unroll
                            for (int j = 0; j < BN / 64; ++j) tma_load_2d(b + j * (64 * BK * 2), &tmB, &full[stage], n_blk * BN + j * 64, kb * BK);
                        }
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (warp-uniform; an elected lane issues) =====================
        {
            constexpr uint32_t idesc = make_idesc(BM, BN, A_MN, B_MN);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
                const int split = tile / (p.m_blocks * p.n_blocks);
                const int kb0 = split * p.kb_per_split, kb1 = min(p.kblocks, kb0 + p.kb_per_split);
                mbar_wait(&tempty[acc], acc_phase ^ 1);
                tcgen05_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tcgen05_fence_after();
                    const uint32_t a0 = smem_u32(sA + stage * A_STAGE), b0 = smem_u32(sB + stage * B_STAGE);
                    if (elect_one_lane()) {
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) {
                            // K-major: 16 bf16 = 32 B inside the 128 B swizzle row; SBO = 8 rows * 128 B.
                            // MN-major: 16 k-rows = 2048 B; LBO = next 64-wide MN atom (64*BK*2 B), SBO = 8 k-rows.
                            const uint64_t da = A_MN ? make_desc(a0 + k * 2048, 64 * BK * 2, 1024) : make_desc(a0 + k * 32, 16, 1024);
                            const uint64_t db = B_MN ? make_desc(b0 + k * 2048, 64 * BK * 2, 1024) : make_desc(b0 + k * 32, 16, 1024);
                            umma_bf16(tmem_d, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
                        }
                        tcgen05_commit(&empty[stage]);      // frees the smem slot when these MMAs retire
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                if (elect_one_lane()) tcgen05_commit(&tfull[acc]);   // accumulator complete -> epilogue
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ===================== epilogue warps (TMEM -> registers -> global) =====================
        const int quad = warp & 3;                          // TMEM lane quadrant this warp may access
        const Epi& e = p.epi;
        int acc = 0; uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
            const int split = tile / (p.m_blocks * p.n_blocks);
            const int rem = tile % (p.m_blocks * p.n_blocks);
            const int m_blk = rem / p.n_blocks, n_blk = rem % p.n_blocks;
            mbar_wait(&tfull[acc], acc_phase);
            tcgen05_fence_after();
            const int m = m_blk * BM + quad * 32 + lane;
            const bool row_ok = m < e.M;
#pragma unroll 1
            for (int c = 0; c < BN / 32; ++c) {
                uint32_t r[32];
                tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + c * 32), r);
                const int n0 = n_blk * BN + c * 32;
                if (row_ok && n0 < e.N) {
                    const bool full32 = n0 + 32 <= e.N;
                    float v[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
                    if (e.bias) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) if (full32 || n0 + j < e.N) v[j] += __ldg(e.bias + n0 + j);
                    }
                    if (e.out_pre) {
                        __nv_bfloat16* dst = e.out_pre + (size_t)m * e.ld_pre + n0;
                        if (full32 && (e.ld_pre & 7) == 0) {
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                uint4 u;
                                __nv_bfloat162 t0 = __floats2bfloat162_rn(v[q * 8 + 0], v[q * 8 + 1]), t1 = __floats2bfloat162_rn(v[q * 8 + 2], v[q * 8 + 3]);
                                __nv_bfloat162 t2 = __floats2bfloat162_rn(v[q * 8 + 4], v[q * 8 + 5]), t3 = __floats2bfloat162_rn(v[q * 8 + 6], v[q * 8 + 7]);
                                u.x = *(uint32_t*)&t0; u.y = *(uint32_t*)&t1; u.z = *(uint32_t*)&t2; u.w = *(uint32_t*)&t3;
                                *reinterpret_cast<uint4*>(dst + q * 8) = u;
                            }
                        } else {
                            for (int j = 0; j < 32; ++j) if (n0 + j < e.N) dst[j] = __float2bfloat16(v[j]);
                        }
                    }
                    if (e.act == 1) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
                    } else if (e.act == 2) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = mish_f(v[j]);
                    }
                    if (e.mask) {
                        const __nv_bfloat16* src = e.mask + (size_t)m * e.ldmask + n0;
                        if (full32 && (e.ldmask & 7) == 0) {
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                uint4 u = *reinterpret_cast<const uint4*>(src + q * 8);
                                const __nv_bfloat16* hb = reinterpret_cast<const __nv_bfloat16*>(&u);
#pragma unroll
                                for (int j = 0; j < 8; ++j) {
                                    float mv = __bfloat162float(hb[j]);
                                    v[q * 8 + j] *= (e.mask_mode == 1) ? (mv > 0.f ? 1.f : 0.f) : mish_grad_f(mv);
                                }
                            }
                        } else {
                            for (int j = 0; j < 32; ++j) if (n0 + j < e.N) {
                                float mv = __bfloat162float(src[j]);
                                v[j] *= (e.mask_mode == 1) ? (mv > 0.f ? 1.f : 0.f) : mish_grad_f(mv);
                            }
                        }
                    }
                    if (e.add) {
                        const __nv_bfloat16* src = e.add + (size_t)m * e.ldadd + n0;
                        if (full32 && (e.ldadd & 7) == 0) {
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                uint4 u = *reinterpret_cast<const uint4*>(src + q * 8);
                                const __nv_bfloat16* hb = reinterpret_cast<const __nv_bfloat16*>(&u);
#pragma unroll
                                for (int j = 0; j < 8; ++j) v[q * 8 + j] += __bfloat162float(hb[j]);
                            }
                        } else {
                            for (int j = 0; j < 32; ++j) if (n0 + j < e.N) v[j] += __bfloat162float(src[j]);
                        }
                    }
                    if (e.out_bf16) {
                        __nv_bfloat16* dst = e.out_bf16 + (size_t)m * e.ld_bf16 + n0;
                        if (full32 && (e.ld_bf16 & 7) == 0) {
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                uint4 u;
                                __nv_bfloat162 t0 = __floats2bfloat162_rn(v[q * 8 + 0], v[q * 8 + 1]), t1 = __floats2bfloat162_rn(v[q * 8 + 2], v[q * 8 + 3]);
                                __nv_bfloat162 t2 = __floats2bfloat162_rn(v[q * 8 + 4], v[q * 8 + 5]), t3 = __floats2bfloat162_rn(v[q * 8 + 6], v[q * 8 + 7]);
                                u.x = *(uint32_t*)&t0; u.y = *(uint32_t*)&t1; u.z = *(uint32_t*)&t2; u.w = *(uint32_t*)&t3;
                                *reinterpret_cast<uint4*>(dst + q * 8) = u;
                            }
                        } else {
                            for (int j = 0; j < 32; ++j) if (n0 + j < e.N) dst[j] = __float2bfloat16(v[j]);
                        }
                    }
                    if (e.out_f32 && e.f32_atomic) {
                        float* dst = e.out_f32 + (size_t)m * e.ld_f32 + n0;
                        if (full32 && (e.ld_f32 & 3) == 0 && ((uintptr_t)dst & 15) == 0) {   // (a net's slice of the flat gradient need not start 16-byte aligned)
#pragma unroll
                            for (int q = 0; q < 8; ++q)
                                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + q * 4), "f"(v[q * 4]), "f"(v[q * 4 + 1]), "f"(v[q * 4 + 2]), "f"(v[q * 4 + 3]) : "memory");
                        } else {
                            for (int j = 0; j < 32; ++j) if (n0 + j < e.N) atomicAdd(dst + j, v[j]);
                        }
                    } else if (e.out_f32) {
                        float* dst = e.out_f32 + (size_t)split * e.split_stride + (size_t)m * e.ld_f32 + n0;
                        if (full32 && (e.ld_f32 & 3) == 0 && ((uintptr_t)dst & 15) == 0) {
#pragma unroll
                            for (int q = 0; q < 8; ++q)
                                *reinterpret_cast<float4*>(dst + q * 4) = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
                        } else {
                            for (int j = 0; j < 32; ++j) if (n0 + j < e.N) dst[j] = v[j];
                        }
                    }
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*encode_fn_t)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static encode_fn_t g_encode = nullptr;

static int load_encode() {
    if (g_encode) return 0;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || !fn || qres != cudaDriverEntryPointSuccess) DPPO_FAIL(-8, "cuTensorMapEncodeTiled is not available from the driver");
    g_encode = (encode_fn_t)fn;
    return 0;
}
// row-major bf16 matrix [rows][cols] with leading dimension ld (elements); box = [box_rows][box_cols]
// A tensor map is a pure function of (address, extents, pitch, box): the programs of a step re-create the same few hundred descriptors
// every call (workspace addresses are stable), and cuTensorMapEncodeTiled costs about a microsecond each - more host time per step than
// all the launches together.  Per-thread cache, dropped wholesale when it grows past 8192 entries.
struct MapKey {
    const void* base; uint64_t rows, cols, ld; uint32_t br, bc;
    bool operator==(const MapKey& o) const { return base == o.base && rows == o.rows && cols == o.cols && ld == o.ld && br == o.br && bc == o.bc; }
};
struct MapKeyHash {
    size_t operator()(const MapKey& k) const {
        uint64_t h = (uint64_t)(uintptr_t)k.base * 0x9E3779B97F4A7C15ull;
        h ^= (k.rows + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2));
        h ^= (k.cols * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2));
        h ^= (k.ld * 0x165667B19E3779F9ull + (h << 6) + (h >> 2));
        h ^= (((uint64_t)k.br << 32 | k.bc) + (h << 6) + (h >> 2));
        return (size_t)h;
    }
};
static int make_map_uncached(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols);
static int make_map(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols) {
    static thread_local std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
    const MapKey k{base, rows, cols, ld, box_rows, box_cols};
    auto it = cache.find(k);
    if (it != cache.end()) { *m = it->second; return 0; }
    DPPO_TRY(make_map_uncached(m, base, rows, cols, ld, box_rows, box_cols));
    if (cache.size() > 8192) cache.clear();
    cache.emplace(k, *m);
    return 0;
}
static int make_map_uncached(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols) {
    DPPO_TRY(load_encode());
    if ((((uintptr_t)base) & 15) || ((ld * 2) & 15)) DPPO_FAIL(-8, "tensor map operand is not 16-byte aligned (ld=%llu)", (unsigned long long)ld);
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * 2};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) DPPO_FAIL(-8, "cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu ld=%llu box=%ux%u", (int)r,
                                     (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_rows, box_cols);
    return 0;
}

// One operand of a GEMM.  K-major: memory is [mn][k] (ld elements between mn rows).
// MN-major: memory is [k][mn].  `mn`/`k` are the logical extents (TMA zero-fills beyond them).
struct Operand { const __nv_bfloat16* ptr; bool mn_major; int64_t mn, k, ld; };

struct Gemm {
    Operand A, A2, B;      // A2.ptr == nullptr: no K concatenation
    int M, N;              // output extents (M rows of A, N rows/cols of B)
    int splits;            // split-K factor (fp32 partial outputs)
    double alg_flops;      // algorithmic flops (un-padded dims) for the live roofline; 0 = use the padded GEMM shape
    Epi epi;
};

template <int BN, bool A_MN, bool B_MN>
static int launch_t(dppo_handle* h, cudaStream_t s, const Gemm& g) {
    CUtensorMap tA, tA2, tB;
    const Operand& A = g.A; const Operand& B = g.B;
    if (!A_MN) DPPO_TRY(make_map(&tA, A.ptr, A.mn, A.k, A.ld, BM, BK)); else DPPO_TRY(make_map(&tA, A.ptr, A.k, A.mn, A.ld, BK, 64));
    if (g.A2.ptr) {
        if (!A_MN) DPPO_TRY(make_map(&tA2, g.A2.ptr, g.A2.mn, g.A2.k, g.A2.ld, BM, BK)); else DPPO_TRY(make_map(&tA2, g.A2.ptr, g.A2.k, g.A2.mn, g.A2.ld, BK, 64));
    } else tA2 = tA;
    if (!B_MN) DPPO_TRY(make_map(&tB, B.ptr, B.mn, B.k, B.ld, BN, BK)); else DPPO_TRY(make_map(&tB, B.ptr, B.k, B.mn, B.ld, BK, 64));
    Params p;
    p.m_blocks = (g.M + BM - 1) / BM; p.n_blocks = (g.N + BN - 1) / BN;
    const int ka = (int)((A.k + BK - 1) / BK), ka2 = g.A2.ptr ? (int)((g.A2.k + BK - 1) / BK) : 0;
    p.kblocks = ka + ka2; p.ka_blocks = ka;
    int splits = g.splits < 1 ? 1 : g.splits;
    if (splits > p.kblocks) splits = p.kblocks;
    p.kb_per_split = (p.kblocks + splits - 1) / splits;
    p.splits = (p.kblocks + p.kb_per_split - 1) / p.kb_per_split;
    p.epi = g.epi;
    auto kern = gemm_kernel<BN, A_MN, B_MN>;
    static bool attr_set_dev[64] = {};      // function attributes are per device
    bool& attr_set = attr_set_dev[h->device & 63];
    if (!attr_set) { CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes<BN>())); attr_set = true; }
    const int tiles = p.m_blocks * p.n_blocks * p.splits;
    const int grid = tiles < h->sm_count ? tiles : h->sm_count;
    prof_begin(h, s);
    kern<<<grid, NUM_THREADS, smem_bytes<BN>(), s>>>(tA, tA2, tB, p);
    prof_end(h, s, g.alg_flops > 0 ? g.alg_flops : 2.0 * (double)g.M * (double)g.N * (double)(A.k + (g.A2.ptr ? g.A2.k : 0)), 1);
    h->launches++; h->tc_launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) DPPO_FAIL(-3, "tc gemm launch failed: %s", cudaGetErrorString(e));
    return p.splits;
}

// returns the number of split-K partials written (>= 1) or a negative error
static int launch(dppo_handle* h, cudaStream_t s, const Gemm& g) {
    const bool a = g.A.mn_major, b = g.B.mn_major;
    const int BN = g.N > 128 ? 256 : (g.N > 64 ? 128 : (g.N > 32 || b ? 64 : 32));
#define TC_DISPATCH(BNV) \
    (a ? (b ? launch_t<BNV, true, true>(h, s, g) : launch_t<BNV, true, false>(h, s, g)) \
       : (b ? launch_t<BNV, false, true>(h, s, g) : launch_t<BNV, false, false>(h, s, g)))
    switch (BN) {
        case 256: return TC_DISPATCH(256);
        case 128: return TC_DISPATCH(128);
        case 64: return TC_DISPATCH(64);
        default: return a ? launch_t<32, true, false>(h, s, g) : launch_t<32, false, false>(h, s, g);
    }
#undef TC_DISPATCH
}

}  // namespace tc

