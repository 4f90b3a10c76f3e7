// Split-precision tcgen05 path (DPPO_PREC_BF16X3): fp32-faithful results on the bf16 tensor pipe.
//
// Every fp32 operand x is carried as bf16 PLANES p0 = bf16(x), p1 = bf16(x - p0), p2 = bf16(x - p0 - p1) (8 mantissa bits
// each) and every product is evaluated as a sum of exact bf16 x bf16 plane products accumulated in fp32 in tensor memory,
// several tcgen05.mma per k-step into ONE accumulator:
//   P = 2 (16-bit operands, backward / weight-gradient GEMMs):  A B ~= A0 B0 + A1 B0 + A0 B1              (dropped: 2^-18)
//   P = 3 (24-bit operands; the first forward version, kept for the debug GEMM entry points and the tests that compare the variants):
//                                                               A B ~= A0 B0 + A0 B1 + A1 B0 + A1 B1 + A0 B2 + A2 B0   (2^-27)
// Why the forward pass needs more than 16 bits: the loss is only piecewise smooth (ReLU kinks, the +-1 clip of x0, the PPO ratio clip).  A
// forward deviation eps from the reference flips about eps * density units across a kink, and every flipped unit switches a
// whole gradient term on or off: the actor-gradient error against the reference grows like sqrt(eps) - 2e-3 of the largest
// entry with 16-bit forward operands (measured, tools/flip_probe.py), against the 1e-3 north_star's fp32 mode is held to.
// With >= 22-bit forward operands the forward pass is as close to the reference as the FFMA path is; the backward and
// weight-gradient GEMMs are smooth in their operands and keep P = 2 (1e-5 relative).
//   F16 (forward GEMMs in front of kinks): the same 22 bits from TWO fp16 planes h0 = fp16(x), h1 = fp16(x - h0) (11 bits each) and
//   three products A0 B0 | A1 B0 + A0 B1 in two accumulators: half the MMAs and two thirds of the operand bytes of P = 3 - these
//   GEMMs are bound by the bytes an SM can take in, not by the tensor pipe.  fp16's narrow exponent is handled by scale: weights are
//   stored as planes of 2^10 w (|w| < 64; a weight of 1e-5 still keeps 11 + 8 bits) and the epilogue multiplies by 2^-10; activations are
//   O(1) and unscaled (below 0.1 the second plane is subnormal: absolute error 3e-8 per element, 2e-8 on a K = 512 output).  Gradients
//   keep bf16 planes (they carry 1/N: fp16 would flush them), and one tcgen05.mma cannot take an fp16 and a bf16 operand (the
//   descriptor has a format field per operand, the hardware traps on a mixed one: measured), so when a backward pass follows the
//   forward epilogue ALSO stores the two bf16 planes of each activation for the weight-gradient GEMMs.
//
//   ts::split_gemm_kernel<BN, A_MN, B_MN, P>   D[M,N] = sum_seg sum_(i,j) A_i B_j
//     * a shared-memory stage holds the 2 P plane tiles of one 64-deep k-block (TMA, 128-byte swizzle): each byte that
//       enters the SM feeds 1.5 (P = 2) or 2 (P = 3) MMAs instead of the 1 of a K-concatenated formulation
//     * 128 x BN accumulators double-buffered in TMEM; 4 epilogue warps write fp32 (+ bias): the narrow output layer and the
//       split-K partials of the weight gradients (deterministic fixed-order reduction).  The layers whose output is the next
//       GEMM's operand run on tsp::pair_gemm_kernel below.
//     * operands K-major or MN-major as stored (activations [rows][features], weights [in][out]): nothing is transposed
//   host programs (the data flow of the per-layer bf16 programs of tc_path.cuh, every activation / gradient as two planes):
//     forward L0, L1 and the folded output layer [a1 | h0] x [W2 W3 ; W0 W3] (block.l2 and the output layer in one narrow
//     GEMM), backward dh1 / du, the four weight-gradient products per net (dW3, dW2 and the residual share of dW0 assembled
//     from a1^T dout / h0^T dout), bias gradients by column sums, the time-embedding backward from dW0's one-hot rows.
#pragma once
#include "tc_path.cuh"

namespace ts {
using namespace tc;

constexpr int SBM = 128, SBK = 64, STHREADS = 192;   // warp 0: TMA, warp 1: MMA + TMEM alloc, warps 2..5: epilogue
constexpr int MAXP = 3;

struct Epi {
    int M, N;                                         // valid extents of the output
    const float* bias;                                // [N]
    float* out_f32; int ld_f32; size_t split_stride;  // fp32 row-major (+ split * split_stride)
    float scale;                                      // F16 kernels: the accumulators are multiplied by this (1 / weight scale)
};
struct Params {
    int m_blocks, n_blocks, splits;
    int kblocks, kb_per_split;                        // K blocks (of 64) in total / per split
    int ka_blocks;                                    // K blocks taken from A segment 0 (the rest from segment 1)
    Epi epi;
};
struct Maps { CUtensorMap a[2][MAXP], b[2][MAXP]; };    // [segment][plane]; k coordinates are local to the segment

// stage = P A-plane tiles + P B-plane tiles of one k-block
template <int BN, int P> __host__ __device__ constexpr int stage_bytes() { return P * (SBM * SBK * 2 + BN * SBK * 2); }
template <int BN, int P> __host__ __device__ constexpr int stages() { return (220 * 1024) / stage_bytes<BN, P>() > 4 ? 4 : (220 * 1024) / stage_bytes<BN, P>(); }
template <int BN, int P> constexpr size_t smem_bytes() { return (size_t)stages<BN, P>() * stage_bytes<BN, P>() + 1024 + 256; }

__device__ __forceinline__ void split_bf16(float v, bf16& hi, bf16& lo) {
    hi = __float2bfloat16(v);
    lo = __float2bfloat16(v - __bfloat162float(hi));
}
__device__ __forceinline__ void split_bf16_3(float v, bf16& p0, bf16& p1, bf16& p2) {
    p0 = __float2bfloat16(v);
    const float r1 = v - __bfloat162float(p0);            // exact
    p1 = __float2bfloat16(r1);
    p2 = __float2bfloat16(r1 - __bfloat162float(p1));     // exact remainder, rounded to the third plane
}
// fp16 planes live in the same 16-bit containers as the bf16 ones (the tensor maps only see 2-byte elements)
__device__ __forceinline__ bf16 f16_bits(float v, float& back) {
    const __half hv = __float2half_rn(v);
    back = __half2float(hv);
    return __ushort_as_bfloat16(__half_as_ushort(hv));
}
__device__ __forceinline__ void split_f16(float v, bf16& hi, bf16& lo) {
    float b0, b1;
    hi = f16_bits(v, b0);
    lo = f16_bits(v - b0, b1);
}
// two values at a time with the packed conversions (F2FP.*.PACK_AB; the scalar __float2bfloat16 compiles to F2F on the quarter-rate
// conversion pipe): hi2 / lo2 hold (a, b) as the low / high 16 bits
__device__ __forceinline__ void split_bf16_pair(float a, float b, uint32_t& hi2, uint32_t& lo2) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    const uint32_t hb = *reinterpret_cast<const uint32_t*>(&h);
    const float ra = a - __uint_as_float(hb << 16), rb = b - __uint_as_float(hb & 0xffff0000u);
    const __nv_bfloat162 l = __floats2bfloat162_rn(ra, rb);
    hi2 = hb; lo2 = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ void split_f16_pair(float a, float b, uint32_t& hi2, uint32_t& lo2) {
    const __half2 h = __floats2half2_rn(a, b);
    const float2 back = __half22float2(h);
    const __half2 l = __floats2half2_rn(a - back.x, b - back.y);
    hi2 = *reinterpret_cast<const uint32_t*>(&h); lo2 = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ float f16_plane_value(bf16 b) { return __half2float(__ushort_as_half(__bfloat16_as_ushort(b))); }
constexpr float F16_WSCALE = 1024.f;     // forward weights are stored as fp16 planes of 2^10 w

template <int BN, bool A_MN, bool B_MN, int P, bool DUAL, bool F16 = false>
__global__ void __launch_bounds__(STHREADS, 1) split_gemm_kernel(const __grid_constant__ Maps maps, const Params p) {
    constexpr int STG = stages<BN, P>();
    constexpr int A_TILE = SBM * SBK * 2, B_TILE = BN * SBK * 2, STAGE = stage_bytes<BN, P>();
    // P = 3: the five correction products go to a SECOND accumulator and are added to the main one (A0 B0) in fp32 registers by
    // the epilogue.  tcgen05 accumulation truncates: every MMA into an accumulator costs up to one ulp of ITS magnitude, biased
    // (measured: 192 accumulations per element at K = 512 left 5e-6 relative whether the operands carried 16 or 24 bits).  The
    // correction sum is 2^-8 of the main one, so its truncations vanish and the main accumulator sees K/16 of them instead of 6 K/16.
    constexpr int NACC = DUAL ? 2 : 1;
    constexpr int ACC_COLS = NACC * BN;
    constexpr int TMEM_COLS = (2 * ACC_COLS <= 32) ? 32 : (2 * ACC_COLS <= 64 ? 64 : (2 * ACC_COLS <= 128 ? 128 : (2 * ACC_COLS <= 256 ? 256 : 512)));
    static_assert(STG >= 2, "a stage must fit twice");
    static_assert(2 * ACC_COLS <= 512, "accumulators exceed tensor memory");
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + STG * STAGE);
    uint64_t* full = bars;                 // [STG]  TMA -> MMA
    uint64_t* empty = bars + STG;          // [STG]  MMA -> TMA
    uint64_t* tfull = bars + 2 * STG;      // [2]    MMA -> epilogue
    uint64_t* tempty = tfull + 2;          // [2]    epilogue -> MMA
    uint32_t* tmem_slot = (uint32_t*)(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles = p.m_blocks * p.n_blocks * p.splits;

    if (warp == 0 && lane == 0) {
        for (int pl = 0; pl < P; ++pl) { tma_prefetch_desc(&maps.a[0][pl]); tma_prefetch_desc(&maps.b[0][pl]); }
        for (int i = 0; i < STG; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
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
        // ===================== TMA producer: the 2 P plane tiles of one k-block per stage =====================
        int stage = 0; uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
            const int split = tile / (p.m_blocks * p.n_blocks);
            const int rem = tile % (p.m_blocks * p.n_blocks);
            const int m_blk = rem / p.n_blocks, n_blk = rem % p.n_blocks;
            const int kb0 = split * p.kb_per_split, kb1 = min(p.kblocks, kb0 + p.kb_per_split);
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(&empty[stage], phase ^ 1);
                if (elect_one_lane()) {
                    mbar_expect_tx(&full[stage], STAGE);
                    uint8_t* sa = smem + stage * STAGE; uint8_t* sb = sa + P * A_TILE;
                    const int seg = kb < p.ka_blocks ? 0 : 1;
                    const int ka = (seg ? kb - p.ka_blocks : kb) * SBK;
#pragma unroll
                    for (int pl = 0; pl < P; ++pl) {
                        uint8_t* a = sa + pl * A_TILE; uint8_t* b = sb + pl * B_TILE;
                        if (!A_MN) tma_load_2d(a, &maps.a[seg][pl], &full[stage], ka, m_blk * SBM);
                        else {
#pragma unroll
                            for (int j = 0; j < SBM / 64; ++j) tma_load_2d(a + j * (64 * SBK * 2), &maps.a[seg][pl], &full[stage], m_blk * SBM + j * 64, ka);
                        }
                        if (!B_MN) tma_load_2d(b, &maps.b[seg][pl], &full[stage], ka, n_blk * BN);
                        else {
#pragma unroll
                            for (int j = 0; j < BN / 64; ++j) tma_load_2d(b + j * (64 * SBK * 2), &maps.b[seg][pl], &full[stage], n_blk * BN + j * 64, ka);
                        }
                    }
                }
                __syncwarp();
                if (++stage == STG) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer: all plane products of a k-step into one accumulator =====================
        constexpr uint32_t idesc = make_idesc(SBM, BN, A_MN, B_MN, !F16, !F16);
        // (A plane, B plane) pairs, small terms first
        constexpr int NPROD = P == 3 ? 6 : 3;
        constexpr int PA[6] = {2, 0, 1, 1, 0, 0}, PB[6] = {0, 2, 1, 0, 1, 0};       // P = 3
        constexpr int QA[3] = {1, 0, 0}, QB[3] = {0, 1, 0};                          // P = 2
        int stage = 0; uint32_t phase = 0;
        int acc = 0; uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
            const int split = tile / (p.m_blocks * p.n_blocks);
            const int kb0 = split * p.kb_per_split, kb1 = min(p.kblocks, kb0 + p.kb_per_split);
            mbar_wait(&tempty[acc], acc_phase ^ 1);
            tcgen05_fence_after();
            const uint32_t tmem_d = tmem_base + (uint32_t)(acc * ACC_COLS);
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(&full[stage], phase);
                tcgen05_fence_after();
                const uint32_t sa = smem_u32(smem + stage * STAGE), sb = sa + P * A_TILE;
                if (elect_one_lane()) {
#pragma unroll
                    for (int k = 0; k < SBK / 16; ++k) {
                        // K-major: 16 bf16 = 32 B inside the 128 B swizzle row; SBO = 8 rows * 128 B.
                        // MN-major: 16 k-rows = 2048 B; LBO = next 64-wide MN atom (64*SBK*2 B), SBO = 8 k-rows.
                        uint64_t da[P], db[P];
#pragma unroll
                        for (int pl = 0; pl < P; ++pl) {
                            da[pl] = A_MN ? make_desc(sa + pl * A_TILE + k * 2048, 64 * SBK * 2, 1024) : make_desc(sa + pl * A_TILE + k * 32, 16, 1024);
                            db[pl] = B_MN ? make_desc(sb + pl * B_TILE + k * 2048, 64 * SBK * 2, 1024) : make_desc(sb + pl * B_TILE + k * 32, 16, 1024);
                        }
#pragma unroll
                        for (int q = 0; q < NPROD; ++q) {
                            const int ia = P == 3 ? PA[q] : QA[q], ib = P == 3 ? PB[q] : QB[q];
                            if (NACC == 2) {       // main product (last in the list) -> columns [0, BN), corrections -> [BN, 2 BN)
                                const bool main = q == NPROD - 1;
                                umma_bf16(tmem_d + (main ? 0u : (uint32_t)BN), da[ia], db[ib], idesc, (kb > kb0 || k > 0 || (!main && q > 0)) ? 1u : 0u);
                            } else umma_bf16(tmem_d, da[ia], db[ib], idesc, (kb > kb0 || k > 0 || q > 0) ? 1u : 0u);
                        }
                    }
                    tcgen05_commit(&empty[stage]);
                }
                __syncwarp();
                if (++stage == STG) { stage = 0; phase ^= 1; }
            }
            if (elect_one_lane()) tcgen05_commit(&tfull[acc]);
            __syncwarp();
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    } else {
        // ===================== epilogue warps (TMEM -> registers -> global planes) =====================
        const int quad = warp & 3;
        const Epi& e = p.epi;
        int acc = 0; uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
            const int split = tile / (p.m_blocks * p.n_blocks);
            const int rem = tile % (p.m_blocks * p.n_blocks);
            const int m_blk = rem / p.n_blocks, n_blk = rem % p.n_blocks;
            mbar_wait(&tfull[acc], acc_phase);
            tcgen05_fence_after();
            const int m = m_blk * SBM + quad * 32 + lane;
            const bool row_ok = m < e.M;
#pragma unroll 1
            for (int c = 0; c < BN / 32; ++c) {
                uint32_t r[32];
                tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * ACC_COLS + c * 32), r);
                float v[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
                if (NACC == 2) {
                    tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * ACC_COLS + BN + c * 32), r);
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] += __uint_as_float(r[j]);
                }
                if (F16) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] *= e.scale;
                }
                const int n0 = n_blk * BN + c * 32;
                if (row_ok && n0 < e.N) {
                    const bool full32 = n0 + 32 <= e.N;
                    const int nvalid = full32 ? 32 : e.N - n0;
                    if (e.bias) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) if (full32 || j < nvalid) v[j] += __ldg(e.bias + n0 + j);
                    }
                    if (e.out_f32) {
                        float* dst = e.out_f32 + (size_t)split * e.split_stride + (size_t)m * e.ld_f32 + n0;
                        if (full32 && (e.ld_f32 & 3) == 0) {
#pragma unroll
                            for (int q = 0; q < 8; ++q)
                                *reinterpret_cast<float4*>(dst + q * 4) = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
                        } else {
                            for (int j = 0; j < nvalid; ++j) dst[j] = v[j];
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
// One split operand: `planes` planes with the same shape.  K-major: memory is [mn][k]; MN-major: memory is [k][mn].
struct Operand { const bf16* p[MAXP]; bool mn_major; int64_t mn, k, ld; };
struct Gemm {
    Operand A, A2, B, B2;  // A2.p[0] == nullptr: no K concatenation; else the K-concatenation [A | A2] x [B ; B2]
    int planes;            // 2 or 3 (every operand must carry that many)
    int dual;              // two planes with the correction products in a second accumulator (forward GEMMs in front of kinks)
    int f16;               // operands are fp16 planes (planes = 2, dual = 1), B scaled by 1 / epi.scale
    int M, N, splits;
    double alg_flops;      // algorithmic flops (un-padded dims, ONE product per MAC) for the live roofline
    Epi epi;
};

template <int BN, bool A_MN, bool B_MN, int P, bool DUAL, bool F16 = false>
static int launch_t(dppo_handle* h, cudaStream_t s, const Gemm& g) {
    Maps mp;
    const Operand& A = g.A; const Operand& B = g.B;
    auto amap = [&](CUtensorMap* m, const bf16* ptr, const Operand& o) -> int {
        return A_MN ? make_map(m, ptr, o.k, o.mn, o.ld, SBK, 64) : make_map(m, ptr, o.mn, o.k, o.ld, SBM, SBK);
    };
    for (int pl = 0; pl < MAXP; ++pl) {
        const int src = pl < P ? pl : 0;
        DPPO_TRY(amap(&mp.a[0][pl], A.p[src], A));
        if (g.A2.p[0]) DPPO_TRY(amap(&mp.a[1][pl], g.A2.p[src], g.A2)); else mp.a[1][pl] = mp.a[0][pl];
        auto bmap = [&](CUtensorMap* m, const bf16* ptr, const Operand& o) -> int {
            return B_MN ? make_map(m, ptr, o.k, o.mn, o.ld, SBK, 64) : make_map(m, ptr, o.mn, o.k, o.ld, BN, SBK);
        };
        DPPO_TRY(bmap(&mp.b[0][pl], B.p[src], B));
        if (g.A2.p[0]) DPPO_TRY(bmap(&mp.b[1][pl], g.B2.p[src], g.B2)); else mp.b[1][pl] = mp.b[0][pl];
    }
    Params p;
    p.m_blocks = (g.M + SBM - 1) / SBM; p.n_blocks = (g.N + BN - 1) / BN;
    const int ka = (int)((A.k + SBK - 1) / SBK), ka2 = g.A2.p[0] ? (int)((g.A2.k + SBK - 1) / SBK) : 0;
    p.kblocks = ka + ka2; p.ka_blocks = ka;
    int splits = g.splits < 1 ? 1 : g.splits;
    if (splits > p.kblocks) splits = p.kblocks;
    p.kb_per_split = (p.kblocks + splits - 1) / splits;
    p.splits = (p.kblocks + p.kb_per_split - 1) / p.kb_per_split;
    p.epi = g.epi;
    auto kern = split_gemm_kernel<BN, A_MN, B_MN, P, DUAL, F16>;
    static bool attr_set_dev[64] = {};      // function attributes are per device
    bool& attr_set = attr_set_dev[h->device & 63];
    if (!attr_set) { CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes<BN, P>())); attr_set = true; }
    const int tiles = p.m_blocks * p.n_blocks * p.splits;
    const int grid = tiles < h->sm_count ? tiles : h->sm_count;
    prof_begin(h, s);
    kern<<<grid, STHREADS, smem_bytes<BN, P>(), s>>>(mp, p);
    prof_end(h, s, g.alg_flops > 0 ? g.alg_flops : 2.0 * (double)g.M * (double)g.N * (double)(A.k + (g.A2.p[0] ? g.A2.k : 0)), 3,
             (P == 3 ? 6.0 : 3.0) * 2.0 * (double)p.m_blocks * SBM * (double)p.n_blocks * BN * (double)p.kblocks * SBK);
    h->launches++; h->tc_launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) DPPO_FAIL(-3, "split gemm launch failed: %s", cudaGetErrorString(e));
    return p.splits;
}
// returns the number of split-K partials written (>= 1) or a negative error.  Only the combinations the programs below use
// are instantiated: forward (K-major A, MN-major B; P = 2 or 3), output layer / backward (K-major both), weight gradients
// (MN-major both, P = 2).
static int launch(dppo_handle* h, cudaStream_t s, const Gemm& g) {
    const bool a = g.A.mn_major, b = g.B.mn_major;
    if (g.f16) {
        if (g.planes == 2 && g.dual && !a && !b && g.N <= 32) return launch_t<32, false, false, 2, true, true>(h, s, g);
        // the folded output layer of an action chunk wider than 32: one 128-wide column block, so the [a1 | h0] rows are read once
        if (g.planes == 2 && g.dual && !a && !b && g.N <= 128) return launch_t<128, false, false, 2, true, true>(h, s, g);
        if (g.planes == 2 && g.dual && !a && b) return launch_t<128, false, true, 2, true, true>(h, s, g);
        DPPO_FAIL(-7, "split gemm: this fp16-plane operand layout is not instantiated");
    }
    if (g.planes == 3) {
        if (!a && b) return launch_t<128, false, true, 3, true>(h, s, g);
        if (!a && !b && g.N <= 32) return launch_t<32, false, false, 3, true>(h, s, g);
        DPPO_FAIL(-7, "split gemm: this 3-plane operand layout is not instantiated");
    }
    if (g.dual) {
        if (!a && b) return launch_t<128, false, true, 2, true>(h, s, g);
        if (!a && !b && g.N <= 32) return launch_t<32, false, false, 2, true>(h, s, g);
        DPPO_FAIL(-7, "split gemm: this dual-accumulator operand layout is not instantiated");
    }
    if (!a && b) return launch_t<256, false, true, 2, false>(h, s, g);
    if (!a && !b) return g.N <= 32 ? launch_t<32, false, false, 2, false>(h, s, g) : launch_t<256, false, false, 2, false>(h, s, g);
    if (a && b) return g.N <= 64 ? launch_t<64, true, true, 2, false>(h, s, g) : launch_t<256, true, true, 2, false>(h, s, g);
    DPPO_FAIL(-7, "split gemm: operand layout (A MN-major, B K-major) is not instantiated");
}
}  // namespace ts

struct SplitT { bf16* p[ts::MAXP]; };
static inline SplitT split_null() { SplitT t; t.p[0] = t.p[1] = t.p[2] = nullptr; return t; }

// =====================================================================================================================
// The same plane GEMM on CTA PAIRS (cta_group::2) with a coalesced epilogue, for the layers whose output is the next GEMM's
// operand (forward L0..L2, backward dv / dh1 / du).  What the single-CTA kernel above measured (ncu launch list,
// profiles/r02_split_v1_launches.txt): it is bound by (a) TMA ingest - 96 KB per k-block for 1536 MMA cycles = 62 B/cycle
// against the ~34 B/cycle an SM takes in - and (b) its thread-per-row epilogue, whose 16-byte stores touch 32 different lines
// per warp instruction (a K = 64 layer took as long as a K = 512 one).  Here
//   * a pair owns a 256 x BNP output tile; each CTA stages its own 128 A rows and HALF of the B tile per plane (P = 2, BNP = 256:
//     64 KB per k-block and CTA = 42 B/cycle; P = 3 with two accumulators, BNP = 128: 72 KB for 1536 cycles);
//   * the leader issues the 256-row tcgen05.mma for the pair, commits are multicast, both CTAs' TMA loads report to the
//     leader's barriers (same scheme as tcp::dw_pair_kernel);
//   * eight epilogue warps per CTA (two per TMEM lane quadrant, 32 columns each) convert a [128][64] column group to bf16
//     planes in shared memory in the 128-byte-swizzled image a TMA store expects, and ONE thread stores each plane with
//     cp.async.bulk.tensor: full-line writes, clipped at the matrix edge by the tensor map;
//   * ReLU derivatives travel as bit masks [rows][N/32] (4 bytes per thread and group instead of re-reading an activation
//     plane), Mish derivatives as two gate planes mish'(pre) written next to the activation by the forward epilogue.
namespace tsp {
using namespace tc;
constexpr int PTHREADS = 320;         // warp 0: TMA, warp 1: MMA (leader) + TMEM alloc, warps 2..9: epilogue
constexpr int SLOT = 16384;           // one [128 rows][64 columns] 16-bit plane tile

struct Epi {
    int M, N;                                              // valid extents of the output
    const float* bias; int act;                            // 0 none, 1 relu, 2 mish
    const uint32_t* mask_in; uint32_t* mask_out; int ldm;  // ReLU bit masks [rows][ldm words]; word j = columns [32 j, 32 j + 32)
    const bf16* gate_in[2]; int ldg;                       // Mish backward: *= gate_in[0] + gate_in[1]
    int out_planes;                                        // 2 or 3 planes stored through maps.out
    int gate_out;                                          // Mish forward: also store mish'(pre-activation) as two planes (maps.gate)
    float* colsum_part; int colsum_ld;                     // bias gradient: per 32-row block column sums of the fp32 result,
                                                           // written to colsum_part[rowblock * colsum_ld + column] (rowblock = row / 32)
    float scale;                                           // F16 kernels: accumulators *= scale (1 / weight scale) before the bias
    int out2;                                              // F16 kernels: also store the result as two bf16 planes (maps.out2)
};
struct Params {
    int m_blocks, n_blocks, kblocks, ka_blocks;
    int stg, nslot, dbuf;            // shared-memory plan (host): load stages, staging slots, two staging buffers of nslot / 2 slots
    int gslot;                       // first of the four slots behind the staging slots that take the gate planes in (Mish backward)
    Epi epi;
};
struct Maps { CUtensorMap a[2][ts::MAXP], b[2][ts::MAXP], out[ts::MAXP], gate[2], out2[2]; };

template <int P, int BNP> __host__ __device__ constexpr int stage_bytes() { return P * (128 * 64 * 2 + (BNP / 2) * 64 * 2); }
// The 227 KB of a CTA are split between load stages and epilogue staging slots per launch.  Measured (50 000 x 512 x 512 layers): a
// third load stage is worth more than a second staging buffer (fp16 forward layer 100 -> 88 us), a second staging buffer more than a
// fourth stage; two stages are the minimum - and all a layer of one or two k-blocks can use: there the second staging buffer comes first.
constexpr int SMEM_BUDGET = 227 * 1024 - 1024 - 256;
static inline void smem_plan(int stage_bytes, int planes_staged, int fixed_slots, int kblocks, int& stg, int& nslot, int& dbuf) {
    const int budget = SMEM_BUDGET - fixed_slots * SLOT;
    const int want = kblocks <= 2 ? 2 : 3;
    nslot = planes_staged; dbuf = 0;
    stg = (budget - nslot * SLOT) / stage_bytes;
    if (stg >= want && (budget - 2 * nslot * SLOT) / stage_bytes >= want) { nslot *= 2; dbuf = 1; stg = (budget - nslot * SLOT) / stage_bytes; }
    if (stg > 4) stg = 4;
}

__device__ __forceinline__ void epi_barrier8() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// launches of consecutive plane GEMMs in one stream overlap the next grid's prologue with the previous grid's last wave
static inline int pdl_attrs(cudaLaunchAttribute* at) {
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[1].val.programmaticStreamSerializationAllowed = 1;
    return 2;
}

template <bool B_MN, int P, bool DUAL, int BNP, bool F16 = false>
__global__ void __launch_bounds__(PTHREADS, 1) pair_gemm_kernel(const __grid_constant__ Maps maps, const Params p) {
    const int STG = p.stg, NSLOT = p.nslot + (p.epi.gate_in[0] ? 4 : 0);
    constexpr int A_TILE = 128 * 64 * 2, B_TILE = (BNP / 2) * 64 * 2, STAGE = stage_bytes<P, BNP>();
    constexpr int NACC = DUAL ? 2 : 1, ACC_COLS = NACC * BNP;
    static_assert(2 * ACC_COLS <= 512, "accumulators exceed tensor memory");
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* slots = smem + STG * STAGE;
    uint64_t* bars = (uint64_t*)(slots + NSLOT * SLOT);
    uint64_t* full = bars;                      // leader's: both CTAs' producers + their TMA bytes
    uint64_t* empty = bars + STG;               // per CTA: multicast commit of the MMAs that read the stage
    uint64_t* tfull = bars + 2 * STG;           // per CTA: multicast commit, accumulator complete
    uint64_t* tempty = tfull + 2;               // leader's: the 16 epilogue warps of the pair drained the accumulator
    uint64_t* gfull = tempty + 2;               // per CTA: the gate planes of a column group arrived (TMA, two buffers)
    uint32_t* tmem_slot = (uint32_t*)(gfull + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = fc::cluster_ctarank();
    const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    const int tiles = p.m_blocks * p.n_blocks;
    pdl_launch_dependents();                    // the next kernel's CTAs may take this SM as soon as this CTA is gone

    if (warp == 0 && lane == 0) {
        for (int pl = 0; pl < P; ++pl) { tma_prefetch_desc(&maps.a[0][pl]); tma_prefetch_desc(&maps.b[0][pl]); }
        for (int i = 0; i < STG; ++i) { mbar_init(&full[i], 2); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 16); mbar_init(&gfull[i], 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fc::cluster_sync_all();                     // barriers of both CTAs initialised before anything remote
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    fc::cluster_sync_all();
    tcgen05_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
    // programmatic dependent launch: this grid may have been scheduled while the previous kernel of the stream was draining (its barriers,
    // tensor memory and tensor-map prefetches above overlap that tail); nothing global is touched before the previous grid has completed
    pdl_wait();

    if (warp == 0) {
        // ---- TMA producer (both CTAs): own 128 A rows, own half of the B tile, every plane; bytes and arrival go to the leader
        int stage = 0; uint32_t phase = 0;
        const uint32_t s_addr = smem_u32(smem), full_addr = smem_u32(full);
        for (int tile = pair; tile < tiles; tile += npairs) {
            const int m_blk = tile / p.n_blocks, n_blk = tile % p.n_blocks;
            const int m0 = m_blk * 256 + (int)rank * 128, n0 = n_blk * BNP + (int)rank * (BNP / 2);
            for (int kb = 0; kb < p.kblocks; ++kb) {
                mbar_wait(&empty[stage], phase ^ 1);
                if (elect_one_lane()) {
                    const uint32_t fb = full_addr + stage * 8;
                    fc::mbar_expect_tx_cluster(fc::mapa_rank0(fb), (uint32_t)STAGE);
                    const uint32_t sa = s_addr + stage * STAGE, sb = sa + P * A_TILE;
                    const int seg = kb < p.ka_blocks ? 0 : 1;
                    const int ka = (seg ? kb - p.ka_blocks : kb) * 64;
#pragma unroll
                    for (int pl = 0; pl < P; ++pl) {
                        fc::tma_load_2d_pair(sa + pl * A_TILE, &maps.a[seg][pl], fb, ka, m0);
                        if (!B_MN) fc::tma_load_2d_pair(sb + pl * B_TILE, &maps.b[seg][pl], fb, ka, n0);
                        else {
#pragma unroll
                            for (int j = 0; j < BNP / 128; ++j) fc::tma_load_2d_pair(sb + pl * B_TILE + j * 8192, &maps.b[seg][pl], fb, n0 + j * 64, ka);
                        }
                    }
                }
                __syncwarp();
                if (++stage == STG) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ---- MMA issuer: the leader only
        if (rank == 0) {
            constexpr uint32_t idesc = make_idesc(256, BNP, false, B_MN, !F16, !F16);
            constexpr int NPROD = P == 3 ? 6 : 3;
            constexpr int PA[6] = {2, 0, 1, 1, 0, 0}, PB[6] = {0, 2, 1, 0, 1, 0};       // P = 3: small terms first, A0 B0 last
            constexpr int QA[3] = {1, 0, 0}, QB[3] = {0, 1, 0};                          // P = 2
            int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
            for (int tile = pair; tile < tiles; tile += npairs) {
                mbar_wait(&tempty[acc], acc_phase ^ 1);
                tcgen05_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * ACC_COLS);
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tcgen05_fence_after();
                    const uint32_t sa = smem_u32(smem + stage * STAGE), sb = sa + P * A_TILE;
                    if (elect_one_lane()) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            uint64_t da[P], db[P];
#pragma unroll
                            for (int pl = 0; pl < P; ++pl) {
                                da[pl] = make_desc(sa + pl * A_TILE + k * 32, 16, 1024);
                                db[pl] = B_MN ? make_desc(sb + pl * B_TILE + k * 2048, 8192, 1024) : make_desc(sb + pl * B_TILE + k * 32, 16, 1024);
                            }
#pragma unroll
                            for (int q = 0; q < NPROD; ++q) {
                                const int ia = P == 3 ? PA[q] : QA[q], ib = P == 3 ? PB[q] : QB[q];
                                if (DUAL) {
                                    const bool main = q == NPROD - 1;
                                    tcp::umma_bf16_pair(tmem_d + (main ? 0u : (uint32_t)BNP), da[ia], db[ib], idesc, (kb > 0 || k > 0 || (!main && q > 0)) ? 1u : 0u);
                                } else tcp::umma_bf16_pair(tmem_d, da[ia], db[ib], idesc, (kb > 0 || k > 0 || q > 0) ? 1u : 0u);
                            }
                        }
                        fc::tcgen05_commit_pair(smem_u32(&empty[stage]));
                    }
                    __syncwarp();
                    if (++stage == STG) { stage = 0; phase ^= 1; }
                }
                if (elect_one_lane()) fc::tcgen05_commit_pair(smem_u32(&tfull[acc]));
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ---- epilogue (both CTAs, 8 warps): own 128 rows x BNP columns in groups of 64 columns
        const int quad = warp & 3, half = (warp - 2) >> 2;
        const int rloc = quad * 32 + lane;
        const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
        const bool store_thread = (warp == 2 && lane == 0);
        const Epi& e = p.epi;
        const uint32_t slot_addr = smem_u32(slots);
        const uint32_t row_off = (uint32_t)rloc * 128u, sw = (uint32_t)(rloc & 7);
        int acc = 0; uint32_t acc_phase = 0;
        const uint32_t tempty_leader = fc::mapa_rank0(smem_u32(tempty));
        // a staging buffer: [out planes | bf16 copies (out2) | gate planes]; with two buffers (p.dbuf) the TMA store of a group overlaps
        // the next group's math
        const uint32_t BUF = (uint32_t)(p.dbuf ? p.nslot / 2 : p.nslot);
        const bool dbuf = p.dbuf != 0;
        const uint32_t o2 = (uint32_t)P, og = o2 + ((F16 && e.out2) ? 2u : 0u);     // slot offsets of the copies / the gates inside a buffer
        uint32_t gcount = 0;
        // Mish backward: the gate planes mish'(pre-activation) of a column group come in by TMA one group ahead of their use (two
        // buffers of two planes; the store thread issues, everyone waits on the buffer's barrier).  A buffer is re-filled after all
        // eight warps have passed the barriers of the group that read it.
        const bool gin = e.gate_in[0] != nullptr;
        auto gate_issue = [&](int t, int g, uint32_t gi) {
            const int mb = t / p.n_blocks, nb = t % p.n_blocks;
            uint64_t* bar = &gfull[gi & 1u];
            uint8_t* dst = slots + (size_t)(p.gslot + 2 * (int)(gi & 1u)) * SLOT;
            mbar_expect_tx(bar, 2 * SLOT);
            tma_load_2d(dst, &maps.gate[0], bar, nb * BNP + g * 64, mb * 256 + (int)rank * 128);
            tma_load_2d(dst + SLOT, &maps.gate[1], bar, nb * BNP + g * 64, mb * 256 + (int)rank * 128);
        };
        if (gin && store_thread && pair < tiles) gate_issue(pair, 0, 0u);
        for (int tile = pair; tile < tiles; tile += npairs) {
            const int m_blk = tile / p.n_blocks, n_blk = tile % p.n_blocks;
            const int row0 = m_blk * 256 + (int)rank * 128, m = row0 + rloc;
            const bool row_ok = m < e.M;
            mbar_wait(&tfull[acc], acc_phase);
            tcgen05_fence_after();
#pragma unroll 1
            for (int g = 0; g < BNP / 64; ++g) {
                const int n0 = n_blk * BNP + g * 64 + half * 32;              // this warp's 32 columns
                if (gin && store_thread) {                                    // next group's gates (this tile's, or the next tile's first)
                    if (g + 1 < BNP / 64) gate_issue(tile, g + 1, gcount + 1u);
                    else if (tile + npairs < tiles) gate_issue(tile + npairs, 0, gcount + 1u);
                }
                uint32_t r[32];
                tmem_ld32(tmem_base + lane_base + (uint32_t)(acc * ACC_COLS + g * 64 + half * 32), r);
                float v[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
                if (DUAL) {
                    tmem_ld32(tmem_base + lane_base + (uint32_t)(acc * ACC_COLS + BNP + g * 64 + half * 32), r);
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] += __uint_as_float(r[j]);
                }
                if (F16) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] *= e.scale;
                }
                if (g == BNP / 64 - 1) {                                      // accumulator drained: hand it back before the math
                    tcgen05_fence_before();
                    __syncwarp();
                    if (lane == 0) fc::mbar_arrive_cluster(tempty_leader + acc * 8);
                }
                const bool col_ok = n0 < e.N;
                if (e.bias && col_ok) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] += __ldg(e.bias + n0 + j);
                }
                float gt[32];
                if (e.act == 1) {
                    if (e.mask_out) {
                        uint32_t bits = 0u;
#pragma unroll
                        for (int j = 0; j < 32; ++j) bits |= (v[j] > 0.f ? 1u : 0u) << j;
                        if (row_ok && col_ok) e.mask_out[(size_t)m * e.ldm + (n0 >> 5)] = bits;
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
                } else if (e.act == 2) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) { float y; fc::mish_and_grad(v[j], y, gt[j]); v[j] = y; }
                }
                if (e.mask_in) {
                    const uint32_t bits = (row_ok && col_ok) ? __ldg(e.mask_in + (size_t)m * e.ldm + (n0 >> 5)) : 0u;
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = ((bits >> j) & 1u) ? v[j] : 0.f;
                }
                if (gin) {
                    mbar_wait(&gfull[gcount & 1u], (gcount >> 1) & 1u);
                    const uint32_t ga = slot_addr + (uint32_t)(p.gslot + 2 * (int)(gcount & 1u)) * SLOT + row_off;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        uint4 uh, ul;
                        const uint32_t off = ((uint32_t)(half * 4 + q) ^ sw) << 4;
                        fc::ld_shared_v4(ga + off, uh.x, uh.y, uh.z, uh.w);
                        fc::ld_shared_v4(ga + SLOT + off, ul.x, ul.y, ul.z, ul.w);
                        const bf16* hb = reinterpret_cast<const bf16*>(&uh); const bf16* lb = reinterpret_cast<const bf16*>(&ul);
#pragma unroll
                        for (int j = 0; j < 8; ++j) v[q * 8 + j] *= __bfloat162float(hb[j]) + __bfloat162float(lb[j]);
                    }
                }
                if (e.colsum_part) {
                    // column sums over this warp's 32 rows by recursive halving: lane j ends with the sum of column n0 + j
                    float cs[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) cs[j] = v[j];
#pragma unroll
                    for (int off = 16; off >= 1; off >>= 1) {
#pragma unroll
                        for (int i = 0; i < off; ++i) {
                            const bool up = (lane & off) != 0;
                            const float send = up ? cs[i] : cs[i + off], keep = up ? cs[i + off] : cs[i];
                            cs[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
                        }
                    }
                    if (col_ok && row0 + quad * 32 < e.M) e.colsum_part[(size_t)((row0 >> 5) + quad) * e.colsum_ld + n0 + lane] = cs[0];
                }
                // the staging slots are free once the TMA stores that last used them have read them
                const uint32_t sbuf = dbuf ? (gcount & 1u) * BUF : 0u;
                ++gcount;
                if (store_thread) { if (dbuf) fc::tma_store_wait_read1(); else fc::tma_store_wait_read(); }
                epi_barrier8();
                const uint32_t c0 = (uint32_t)(half * 4);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const uint32_t off = row_off + (((c0 + (uint32_t)q) ^ sw) << 4);
                    if (P == 3) {
                        __align__(16) bf16 t[ts::MAXP][8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) ts::split_bf16_3(v[q * 8 + j], t[0][j], t[1][j], t[2][j]);
#pragma unroll
                        for (int pl = 0; pl < P; ++pl) {
                            const uint4 u = *reinterpret_cast<const uint4*>(t[pl]);
                            fc::st_shared_v4(slot_addr + (sbuf + pl) * SLOT + off, u.x, u.y, u.z, u.w);
                        }
                    } else {
                        uint32_t hi[4], lo[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            if (F16) ts::split_f16_pair(v[q * 8 + 2 * j], v[q * 8 + 2 * j + 1], hi[j], lo[j]);
                            else ts::split_bf16_pair(v[q * 8 + 2 * j], v[q * 8 + 2 * j + 1], hi[j], lo[j]);
                        }
                        fc::st_shared_v4(slot_addr + sbuf * SLOT + off, hi[0], hi[1], hi[2], hi[3]);
                        fc::st_shared_v4(slot_addr + (sbuf + 1) * SLOT + off, lo[0], lo[1], lo[2], lo[3]);
                    }
                    if (F16 && e.out2) {
                        uint32_t hi[4], lo[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j) ts::split_bf16_pair(v[q * 8 + 2 * j], v[q * 8 + 2 * j + 1], hi[j], lo[j]);
                        fc::st_shared_v4(slot_addr + (sbuf + o2) * SLOT + off, hi[0], hi[1], hi[2], hi[3]);
                        fc::st_shared_v4(slot_addr + (sbuf + o2 + 1) * SLOT + off, lo[0], lo[1], lo[2], lo[3]);
                    }
                    if (e.gate_out) {
                        uint32_t hi[4], lo[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j) ts::split_bf16_pair(gt[q * 8 + 2 * j], gt[q * 8 + 2 * j + 1], hi[j], lo[j]);
                        fc::st_shared_v4(slot_addr + (sbuf + og) * SLOT + off, hi[0], hi[1], hi[2], hi[3]);
                        fc::st_shared_v4(slot_addr + (sbuf + og + 1) * SLOT + off, lo[0], lo[1], lo[2], lo[3]);
                    }
                }
                fc::fence_async_smem();
                epi_barrier8();
                if (store_thread) {
                    const int col = n_blk * BNP + g * 64;
                    if (col < e.N) {
                        for (int pl = 0; pl < e.out_planes; ++pl) fc::tma_store_2d(&maps.out[pl], slots + (sbuf + pl) * SLOT, col, row0);
                        if (F16 && e.out2) { fc::tma_store_2d(&maps.out2[0], slots + (sbuf + o2) * SLOT, col, row0); fc::tma_store_2d(&maps.out2[1], slots + (sbuf + o2 + 1) * SLOT, col, row0); }
                        if (e.gate_out) { fc::tma_store_2d(&maps.gate[0], slots + (sbuf + og) * SLOT, col, row0); fc::tma_store_2d(&maps.gate[1], slots + (sbuf + og + 1) * SLOT, col, row0); }
                    }
                    fc::tma_store_commit();
                }
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (store_thread) fc::tma_store_wait_all();
    }
    tcgen05_fence_before();
    __syncthreads();
    fc::cluster_sync_all();                     // the peer may still be signalling our barriers / reading our B halves
    if (warp == 1) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// output planes [M][N] (leading dimension ld) written by TMA; gate planes likewise
struct Gemm {
    ts::Operand A, A2, B, B2;      // A K-major; B K-major or MN-major; [A | A2] x [B ; B2] when A2.p[0] != nullptr
    int planes, dual;              // 2 (single accumulator) or 3 with dual = 1
    int f16;                       // fp16 planes in and out (planes = 2, dual = 1); B carries the weight scale, epi.scale its inverse
    int M, N;
    bf16* out[ts::MAXP]; int ld_out;
    bf16* gate[2];
    bf16* out2[2];                 // f16 only: bf16 copies of the output planes (epi.out2)
    double alg_flops;
    Epi epi;
};

template <bool B_MN, int P, bool DUAL, int BNP, bool F16 = false>
static int launch_t(dppo_handle* h, cudaStream_t s, const Gemm& g) {
    Maps mp;
    for (int pl = 0; pl < ts::MAXP; ++pl) {
        const int src = pl < P ? pl : 0;
        DPPO_TRY(make_map(&mp.a[0][pl], g.A.p[src], g.A.mn, g.A.k, g.A.ld, 128, 64));
        if (g.A2.p[0]) DPPO_TRY(make_map(&mp.a[1][pl], g.A2.p[src], g.A2.mn, g.A2.k, g.A2.ld, 128, 64)); else mp.a[1][pl] = mp.a[0][pl];
        auto bmap = [&](CUtensorMap* m, const bf16* ptr, const ts::Operand& o) -> int {
            return B_MN ? make_map(m, ptr, o.k, o.mn, o.ld, 64, 64) : make_map(m, ptr, o.mn, o.k, o.ld, BNP / 2, 64);
        };
        DPPO_TRY(bmap(&mp.b[0][pl], g.B.p[src], g.B));
        if (g.A2.p[0]) DPPO_TRY(bmap(&mp.b[1][pl], g.B2.p[src], g.B2)); else mp.b[1][pl] = mp.b[0][pl];
        DPPO_TRY(make_map(&mp.out[pl], g.out[pl < g.epi.out_planes ? pl : 0], g.M, g.N, g.ld_out, 128, 64));
    }
    for (int i = 0; i < 2; ++i) {
        if (g.epi.gate_out) DPPO_TRY(make_map(&mp.gate[i], g.gate[i], g.M, g.N, g.ld_out, 128, 64));
        else if (g.epi.gate_in[0]) DPPO_TRY(make_map(&mp.gate[i], g.epi.gate_in[i], g.M, g.N, g.epi.ldg, 128, 64));
        else mp.gate[i] = mp.out[0];
        if (g.epi.out2) DPPO_TRY(make_map(&mp.out2[i], g.out2[i], g.M, g.N, g.ld_out, 128, 64)); else mp.out2[i] = mp.out[0];
    }
    if (g.epi.out2 && !F16) DPPO_FAIL(-7, "split gemm (pair): bf16 copies are an option of the fp16-plane kernel");
    Params p;
    p.m_blocks = (g.M + 255) / 256; p.n_blocks = (g.N + BNP - 1) / BNP;
    const int ka = (int)((g.A.k + 63) / 64), ka2 = g.A2.p[0] ? (int)((g.A2.k + 63) / 64) : 0;
    p.kblocks = ka + ka2; p.ka_blocks = ka;
    p.epi = g.epi;
    if (g.epi.gate_out && g.epi.gate_in[0]) DPPO_FAIL(-7, "split gemm (pair): gate planes go out (forward) or come in (backward), not both");
    smem_plan(stage_bytes<P, BNP>(), P + (g.epi.out2 ? 2 : 0) + (g.epi.gate_out ? 2 : 0), g.epi.gate_in[0] ? 4 : 0, p.kblocks, p.stg, p.nslot, p.dbuf);
    p.gslot = p.nslot;
    if (p.stg < 2 || g.epi.out_planes > P) DPPO_FAIL(-7, "split gemm (pair): shared-memory plan does not fit (%d stages, %d slots)", p.stg, p.nslot);
    const size_t smem_bytes = (size_t)p.stg * stage_bytes<P, BNP>() + (size_t)(p.nslot + (g.epi.gate_in[0] ? 4 : 0)) * SLOT + 1024 + 256;
    auto kern = pair_gemm_kernel<B_MN, P, DUAL, BNP, F16>;
    static bool attr_set_dev[64] = {};      // function attributes are per device
    bool& attr_set = attr_set_dev[h->device & 63];
    if (!attr_set) { CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); attr_set = true; }
    const int tiles = p.m_blocks * p.n_blocks, npairs = h->sm_count / 2;
    const int grid = 2 * (tiles < npairs ? tiles : npairs);
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
    cudaLaunchAttribute at[2];
    cfg.attrs = at; cfg.numAttrs = pdl_attrs(at); cfg.blockDim = dim3(PTHREADS); cfg.gridDim = dim3(grid); cfg.dynamicSmemBytes = smem_bytes; cfg.stream = s;
    prof_begin(h, s);
    cudaError_t le = cudaLaunchKernelEx(&cfg, kern, mp, p);
    prof_end(h, s, g.alg_flops > 0 ? g.alg_flops : 2.0 * (double)g.M * (double)g.N * (double)(g.A.k + (g.A2.p[0] ? g.A2.k : 0)), 0,
             (P == 3 ? 6.0 : 3.0) * 2.0 * (double)p.m_blocks * 256.0 * (double)p.n_blocks * BNP * (double)p.kblocks * 64.0);
    h->launches++; h->tc_launches++;
    if (le != cudaSuccess) DPPO_FAIL(-3, "split gemm (pair) launch failed: %s", cudaGetErrorString(le));
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) DPPO_FAIL(-3, "split gemm (pair) launch failed: %s", cudaGetErrorString(e));
    return 0;
}
static int launch(dppo_handle* h, cudaStream_t s, const Gemm& g) {
    const bool b = g.B.mn_major;
    if (g.f16) {
        if (g.planes == 2 && g.dual) return b ? launch_t<true, 2, true, 128, true>(h, s, g) : launch_t<false, 2, true, 128, true>(h, s, g);
        DPPO_FAIL(-7, "split gemm (pair): fp16 planes need two planes and two accumulators");
    }
    if (g.planes == 3 && g.dual) return b ? launch_t<true, 3, true, 128>(h, s, g) : launch_t<false, 3, true, 128>(h, s, g);
    if (g.planes == 2 && !g.dual) return b ? launch_t<true, 2, false, 256>(h, s, g) : launch_t<false, 2, false, 256>(h, s, g);
    DPPO_FAIL(-7, "split gemm (pair): plane / accumulator combination not instantiated");
}

// ---------------------------------------------------------------------------------------------------------------------
// Grouped weight-gradient GEMM on CTA pairs, two planes per operand:  out_p = X_p^T D_p (+ X2_p^T D2_p)  for up to 10 problems in
// ONE launch (the plane version of tcp::dw_pair_kernel, same wave-balanced K splits).  Every (output tile, K split) item writes
// its fp32 partial tile; dw_reduce_kernel sums an output's partials in a fixed order, so the gradients are bit-reproducible.
constexpr int DSTAGES = 3, DMAXP = 10, DMAPS = 12;
struct DwProb {
    int m_blocks, n_blocks, nb_cta;   // 256-row output blocks; column blocks of nb_cta * 128; 64-column D boxes per CTA per k-block
    int splits, kb_per_split, item_begin;
    int kb_seg0, kb_total;            // k-blocks of the first (X, D) segment / in total (second segment: maps[map2])
    int map2;
    int M_valid, N_valid, ld_out, transposed;
    float* out;
};
struct DwParams { int nprob, items; float* part; DwProb p[DMAXP]; };
struct DwMaps { CUtensorMap a[DMAPS][2], b[DMAPS][2]; };
constexpr size_t dw_smem_bytes() { return (size_t)DSTAGES * 65536 + 1024 + 256; }

__global__ void __launch_bounds__(NUM_THREADS, 1) dw_pair_kernel(const __grid_constant__ DwMaps maps, const DwParams gp) {
    constexpr int A_TILE = 128 * 64 * 2, B_TILE = 128 * 64 * 2, STAGE = 2 * (A_TILE + B_TILE);
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + DSTAGES * STAGE);
    uint64_t* full = bars; uint64_t* empty = bars + DSTAGES; uint64_t* tfull = bars + 2 * DSTAGES; uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = (uint32_t*)(tempty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = fc::cluster_ctarank();
    const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    pdl_launch_dependents();

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < DSTAGES; ++i) { mbar_init(&full[i], 2); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fc::cluster_sync_all();
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    fc::cluster_sync_all();
    tcgen05_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
    pdl_wait();

    auto decode = [&](int item, int& pi, int& m_blk, int& n_blk, int& split) {
        pi = 0;
        while (pi + 1 < gp.nprob && item >= gp.p[pi + 1].item_begin) ++pi;
        const DwProb& P = gp.p[pi];
        const int local = item - P.item_begin, per = P.m_blocks * P.n_blocks;
        split = local / per; const int rem = local % per;
        m_blk = rem / P.n_blocks; n_blk = rem % P.n_blocks;
    };

    if (warp == 0) {
        int stage = 0; uint32_t phase = 0;
        const uint32_t s_addr = smem_u32(smem), full_addr = smem_u32(full);
        for (int item = pair; item < gp.items; item += npairs) {
            int pi, m_blk, n_blk, split; decode(item, pi, m_blk, n_blk, split);
            const DwProb& P = gp.p[pi];
            const int kb0 = split * P.kb_per_split, kb1 = min(P.kb_total, kb0 + P.kb_per_split);
            const uint32_t tx = (uint32_t)(2 * (A_TILE + P.nb_cta * 64 * 64 * 2));
            const int m0 = m_blk * 256 + (int)rank * 128, n0 = n_blk * (P.nb_cta * 128) + (int)rank * (P.nb_cta * 64);
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(&empty[stage], phase ^ 1);
                if (elect_one_lane()) {
                    const uint32_t fb = full_addr + stage * 8;
                    fc::mbar_expect_tx_cluster(fc::mapa_rank0(fb), tx);
                    const int mi = kb < P.kb_seg0 ? pi : P.map2;
                    const int kr = (kb < P.kb_seg0 ? kb : kb - P.kb_seg0) * 64;
#pragma unroll
                    for (int pl = 0; pl < 2; ++pl) {
                        const uint32_t a = s_addr + stage * STAGE + pl * A_TILE, b = s_addr + stage * STAGE + 2 * A_TILE + pl * B_TILE;
                        fc::tma_load_2d_pair(a, &maps.a[mi][pl], fb, m0, kr);
                        fc::tma_load_2d_pair(a + 8192, &maps.a[mi][pl], fb, m0 + 64, kr);
                        for (int j = 0; j < P.nb_cta; ++j) fc::tma_load_2d_pair(b + j * 8192, &maps.b[mi][pl], fb, n0 + j * 64, kr);
                    }
                }
                __syncwarp();
                if (++stage == DSTAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (rank == 0) {
            int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
            for (int item = pair; item < gp.items; item += npairs) {
                int pi, m_blk, n_blk, split; decode(item, pi, m_blk, n_blk, split);
                const DwProb& P = gp.p[pi];
                const int kb0 = split * P.kb_per_split, kb1 = min(P.kb_total, kb0 + P.kb_per_split);
                const uint32_t idesc = make_idesc(256, P.nb_cta * 128, true, true);
                mbar_wait(&tempty[acc], acc_phase ^ 1);
                tcgen05_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * 256);
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tcgen05_fence_after();
                    const uint32_t a0 = smem_u32(smem + stage * STAGE), b0 = a0 + 2 * A_TILE;
                    if (elect_one_lane()) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const uint64_t da0 = make_desc(a0 + k * 2048, 8192, 1024), da1 = make_desc(a0 + A_TILE + k * 2048, 8192, 1024);
                            const uint64_t db0 = make_desc(b0 + k * 2048, 8192, 1024), db1 = make_desc(b0 + B_TILE + k * 2048, 8192, 1024);
                            tcp::umma_bf16_pair(tmem_d, da1, db0, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
                            tcp::umma_bf16_pair(tmem_d, da0, db1, idesc, 1u);
                            tcp::umma_bf16_pair(tmem_d, da0, db0, idesc, 1u);
                        }
                        fc::tcgen05_commit_pair(smem_u32(&empty[stage]));
                    }
                    __syncwarp();
                    if (++stage == DSTAGES) { stage = 0; phase ^= 1; }
                }
                if (elect_one_lane()) fc::tcgen05_commit_pair(smem_u32(&tfull[acc]));
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // epilogue (both CTAs): own 128 rows x the N tile of the item's partial [256][256] fp32
        const int quad = warp & 3;
        int acc = 0; uint32_t acc_phase = 0;
        const uint32_t tempty_leader = fc::mapa_rank0(smem_u32(tempty));
        for (int item = pair; item < gp.items; item += npairs) {
            int pi, m_blk, n_blk, split; decode(item, pi, m_blk, n_blk, split);
            const DwProb& P = gp.p[pi];
            mbar_wait(&tfull[acc], acc_phase);
            tcgen05_fence_after();
            float* dst = gp.part + (size_t)item * 65536 + (size_t)((int)rank * 128 + quad * 32 + lane) * 256;
            const int ntile = P.nb_cta * 128;
#pragma unroll 1
            for (int c = 0; c < ntile / 32; ++c) {
                uint32_t r[32];
                tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * 256 + c * 32), r);
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    *reinterpret_cast<float4*>(dst + c * 32 + q * 4) = make_float4(__uint_as_float(r[q * 4]), __uint_as_float(r[q * 4 + 1]), __uint_as_float(r[q * 4 + 2]), __uint_as_float(r[q * 4 + 3]));
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) fc::mbar_arrive_cluster(tempty_leader + acc * 8);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    fc::cluster_sync_all();
    if (warp == 1) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}
// out[m][n] (or out[n][m] when transposed) = sum over the problem's K splits of its partial tiles, in split order
__global__ void __launch_bounds__(256) dw_reduce_kernel(const DwParams gp, const int* __restrict__ elem_begin) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int pi = 0;
    while (pi + 1 < gp.nprob && i >= elem_begin[pi + 1]) ++pi;
    if (i >= elem_begin[gp.nprob]) return;
    const DwProb& P = gp.p[pi];
    const int local = i - elem_begin[pi];
    // the fastest index follows the output's memory order
    const int m = P.transposed ? local % P.M_valid : local / P.N_valid, n = P.transposed ? local / P.M_valid : local % P.N_valid;
    const int ntile = P.nb_cta * 128, per = P.m_blocks * P.n_blocks;
    const int tile = (m >> 8) * P.n_blocks + n / ntile;
    const float* src = gp.part + (size_t)(P.item_begin + tile) * 65536 + (size_t)(m & 255) * 256 + (n % ntile);
    float acc = 0.f;
    for (int sidx = 0; sidx < P.splits; ++sidx) acc += src[(size_t)sidx * per * 65536];
    if (P.transposed) P.out[(size_t)n * P.ld_out + m] = acc; else P.out[(size_t)m * P.ld_out + n] = acc;
}

// one problem: out = X^T D (+ X2^T D2), X [rows][M], D [rows][Nd] (two planes each); transposed: out[n][m] (ld_out = row length of that layout)
struct DwDesc { SplitT X; int M; SplitT D; int Nd; SplitT X2, D2; float* out; int M_valid, N_valid, ld_out, transposed; double alg_flops; };

static int launch_dw_pair(dppo_handle* h, cudaStream_t s, const DwDesc* d, int n, int rows, float* part, size_t part_floats, int* elem_begin_dev) {
    if (n < 1 || n > DMAXP) DPPO_FAIL(-1, "launch_dw_pair: bad problem count %d", n);
    DwMaps maps; DwParams gp; memset(&gp, 0, sizeof(gp));
    gp.nprob = n; gp.part = part;
    const int kblocks = (rows + 63) / 64;
    const int npairs = h->sm_count / 2;
    double w[DMAXP]; int tiles[DMAXP]; int nmap = n;
    for (int i = 0; i < n; ++i) {
        DwProb& P = gp.p[i];
        if (d[i].M % 64 || d[i].Nd % 64) DPPO_FAIL(-7, "launch_dw_pair: operand widths must be multiples of 64");
        for (int pl = 0; pl < 2; ++pl) {
            DPPO_TRY(make_map(&maps.a[i][pl], d[i].X.p[pl], rows, d[i].M, d[i].M, 64, 64));
            DPPO_TRY(make_map(&maps.b[i][pl], d[i].D.p[pl], rows, d[i].Nd, d[i].Nd, 64, 64));
        }
        P.kb_seg0 = kblocks; P.kb_total = kblocks; P.map2 = i;
        if (d[i].X2.p[0]) {
            if (nmap >= DMAPS) DPPO_FAIL(-7, "launch_dw_pair: too many second segments");
            for (int pl = 0; pl < 2; ++pl) {
                DPPO_TRY(make_map(&maps.a[nmap][pl], d[i].X2.p[pl], rows, d[i].M, d[i].M, 64, 64));
                DPPO_TRY(make_map(&maps.b[nmap][pl], d[i].D2.p[pl], rows, d[i].Nd, d[i].Nd, 64, 64));
            }
            P.map2 = nmap++; P.kb_total = 2 * kblocks;
        }
        P.m_blocks = (d[i].M + 255) / 256;
        const int nb64 = (d[i].Nd + 63) / 64;
        P.nb_cta = nb64 <= 2 ? 1 : 2;
        P.n_blocks = (nb64 + 2 * P.nb_cta - 1) / (2 * P.nb_cta);
        P.M_valid = d[i].M_valid; P.N_valid = d[i].N_valid; P.ld_out = d[i].ld_out; P.out = d[i].out; P.transposed = d[i].transposed;
        tiles[i] = P.m_blocks * P.n_blocks;
        w[i] = (P.nb_cta == 2 ? 1.0 : 0.75) * P.kb_total;              // k-block time of a 128-wide tile: 48 KB staged per CTA instead of 64 KB
    }
    for (int i = nmap; i < DMAPS; ++i) for (int pl = 0; pl < 2; ++pl) { maps.a[i][pl] = maps.a[0][0]; maps.b[i][pl] = maps.b[0][0]; }
    // K splits: the smallest per-item budget for which all items fit the pairs in ONE wave (bisection), at least 4 k-blocks per item
    auto items_for = [&](double budget) { int it = 0; for (int i = 0; i < n; ++i) { int sp = (int)ceil(w[i] / budget); if (sp < 1) sp = 1; it += tiles[i] * sp; } return it; };
    double lo = 4.0, hi = 2.0 * kblocks;
    if (items_for(lo) <= npairs) hi = lo;
    for (int it = 0; it < 40 && hi - lo > 0.25; ++it) { const double mid = 0.5 * (lo + hi); if (items_for(mid) <= npairs) hi = mid; else lo = mid; }
    int items = 0; double flops = 0; int eb[DMAXP + 1];
    eb[0] = 0;
    for (int i = 0; i < n; ++i) {
        DwProb& P = gp.p[i];
        int splits = (int)ceil(w[i] / hi);
        if (splits < 1) splits = 1;
        if (splits > P.kb_total) splits = P.kb_total;
        P.kb_per_split = (P.kb_total + splits - 1) / splits;
        P.splits = (P.kb_total + P.kb_per_split - 1) / P.kb_per_split;
        P.item_begin = items; items += tiles[i] * P.splits;
        flops += d[i].alg_flops;
        eb[i + 1] = eb[i] + P.M_valid * P.N_valid;
    }
    gp.items = items;
    if ((size_t)items * 65536 > part_floats) DPPO_FAIL(-7, "launch_dw_pair: partial buffer too small (%d items)", items);
    CUDA_TRY(cudaMemcpyAsync(elem_begin_dev, eb, (n + 1) * sizeof(int), cudaMemcpyHostToDevice, s));
    static bool attr_set_dev[64] = {};      // function attributes are per device
    bool& attr_set = attr_set_dev[h->device & 63];
    if (!attr_set) { CUDA_TRY(cudaFuncSetAttribute(dw_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dw_smem_bytes())); attr_set = true; }
    const int grid = 2 * (items < npairs ? items : npairs);
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
    cudaLaunchAttribute at[2];
    cfg.attrs = at; cfg.numAttrs = pdl_attrs(at); cfg.blockDim = dim3(NUM_THREADS); cfg.gridDim = dim3(grid); cfg.dynamicSmemBytes = dw_smem_bytes(); cfg.stream = s;
    prof_begin(h, s);
    cudaError_t le = cudaLaunchKernelEx(&cfg, dw_pair_kernel, maps, gp);
    double exec = 0;
    for (int i = 0; i < n; ++i) exec += 3.0 * 2.0 * 256.0 * (double)(gp.p[i].nb_cta * 128) * 64.0 * (double)gp.p[i].kb_total * (double)(gp.p[i].m_blocks * gp.p[i].n_blocks);
    prof_end(h, s, flops, 1, exec);
    h->launches++; h->tc_launches++;
    if (le != cudaSuccess) DPPO_FAIL(-3, "grouped dW (plane pair) launch failed: %s", cudaGetErrorString(le));
    dw_reduce_kernel<<<(eb[n] + 255) / 256, 256, 0, s>>>(gp, elem_begin_dev);
    h->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) DPPO_FAIL(-3, "grouped dW (plane pair) launch failed: %s", cudaGetErrorString(e));
    return 0;
}
}  // namespace tsp

// =====================================================================================================================
// state: plane copies of the weights per net: two bf16 planes (backward GEMMs; forward of a smooth net) and two fp16 planes of
// 2^10 w (forward GEMMs of a net with kinks behind it)
struct TsW { bf16* p[ts::MAXP]; };
struct TsNetW {
    TsW w0, w1;                           // [KP0][H] W0 rows in h0 order, [H][H] W1
    TsW fw0, fw1;                         // fp16 planes, scaled by ts::F16_WSCALE
    TsW ffold;                            // [NOP][H + KP0] planes of [W2 W3 ; W0 W3]^T (fp16 x 2^10 when the net's forward runs on fp16 planes, else
                                          // bf16): the folded output layer, out = [a1 | h0] [W2 W3 ; W0 W3] + bfold
    float* bfold;                         // [NOP]  (b2 (+ b_in)) W3 + b3
    TsW w23p;                             // [H][128] bf16 planes of W2 W3 (columns >= NO zero): dh1 = (dout (W2 W3)^T) . act'(h1) without forming dv
};
struct TsState { TsNetW net[4]; int KP0; int fold_dirty[4]; char* dw3_buf; size_t dw3_bytes; };
// NOP: the padded width of a net's output (gradient seeds dout [N][NOP], rows of ffold / bfold, K of dh1 = dout (W2 W3)^T).  64 up to 32
// outputs; an actor with a wider action chunk (up to 128) takes 128.  The critic (one output) keeps 64.
static inline int ts_nop(int NO) { return NO <= 32 ? 64 : 128; }

static void mark_weights_changed(dppo_handle* h, int net) {
    h->w0p_dirty[net] = 1; h->w23_dirty[net] = 1;
    if (h->ts) h->ts->fold_dirty[net] = 1;
}

__device__ __forceinline__ void ts_put(const TsW& W, size_t i, float v) {
    bf16 a, b; ts::split_bf16(v, a, b);
    W.p[0][i] = a; W.p[1][i] = b;
}
__device__ __forceinline__ void ts_put_f16(const TsW& W, size_t i, float v) {
    bf16 a, b; ts::split_f16(v * ts::F16_WSCALE, a, b);
    W.p[0][i] = a; W.p[1][i] = b;
}
__device__ __forceinline__ void ts_put2(const TsW& W, const TsW& F, size_t i, float v) { ts_put(W, i, v); ts_put_f16(F, i, v); }
// W0 in tc_pack_actor_body's h0 row order and W1, each as two bf16 planes and two fp16 planes; no transposed copy (the backward GEMM
// reads W1 K-major as stored).  W2 and W3 enter the GEMMs only through the folded output layer (ts_fold_kernel).
__global__ void ts_pack_actor_kernel(const float* __restrict__ w, ActorOff o, int A, int td, int Do, int T, int H, int KP0,
                                     const float* __restrict__ bt, const TsNetW W) {
    const size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = i0; i < (size_t)H * H; i += stride) ts_put2(W.w1, W.fw1, i, w[o.w1 + i]);
    for (size_t i = i0; i < (size_t)KP0 * H; i += stride) {
        const int k = (int)(i / H), c = (int)(i % H);
        float v = 0.f;
        if (k < A) v = w[o.win + (size_t)k * H + c];
        else if (k < A + Do) v = w[o.win + (size_t)(k + td) * H + c];
        else if (k < A + Do + T) v = bt[(size_t)(k - A - Do) * H + c];
        ts_put2(W.w0, W.fw0, i, v);
    }
}
__global__ void ts_pack_critic_kernel(const float* __restrict__ w, CriticOff o, int A, int Do, int Hc, int KP0, const TsNetW W) {
    const size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = i0; i < (size_t)Hc * Hc; i += stride) ts_put2(W.w1, W.fw1, i, w[o.w1 + i]);
    for (size_t i = i0; i < (size_t)KP0 * Hc; i += stride) {
        const int k = (int)(i / Hc), c = (int)(i % Hc);
        ts_put2(W.w0, W.fw0, i, (k >= A && k < A + Do) ? w[o.win + (size_t)(k - A) * Hc + c] : 0.f);
    }
}
// h0[r] = [x[r] | obs[r / obs_div] | onehot(t_r) | 1 | 0..] (tc_pack_h0_kernel's layout) as two fp16 planes (hf, when given) and / or two
// bf16 planes (hb, when given); one thread per 8 columns
// flat != nullptr (index-driven minibatch, train_ppo_diffusion_agent.py:292-312 without materialising it): row r is the (rollout row b,
// denoising index k) pair of flat[r] = b * flatK + k: x = chains[b][k], obs = obs[b], t = flatK - 1 - k; bad indices raise *bad and read row 0
__global__ void ts_pack_h0_kernel(const float* __restrict__ x, const float* __restrict__ obs, const int* __restrict__ trow, int tconst,
                                  int N, int A, int Do, int T, int KP0, int obs_div, const SplitT hf, const SplitT hb, int chainK,
                                  const int* __restrict__ flat = nullptr, int flatK = 1, long long flatP = 0, int* __restrict__ bad = nullptr) {
    const int g8 = KP0 / 8;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * g8) return;
    const int r = (int)(i / g8), k0 = (int)(i % g8) * 8;
    int t = trow ? (tconst < 0 ? -tconst - 1 - trow[r] : trow[r]) : tconst;
    size_t xrow = chainK > 0 ? (size_t)(r / chainK) * (chainK + 1) + (r % chainK) : (size_t)r;
    size_t orow = (size_t)(r / obs_div);
    if (flat) {
        int f = flat[r];
        if (f < 0 || (long long)f >= flatP * flatK) { if (bad && k0 == 0) atomicOr(bad, 1); f = 0; }
        const int b = f / flatK, k = f % flatK;
        xrow = (size_t)b * (flatK + 1) + k; orow = (size_t)b; t = flatK - 1 - k;
    }
    __align__(16) bf16 o3[4][8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int k = k0 + j;
        float v = 0.f;
        if (k < A) v = x ? x[xrow * A + k] : 0.f;
        else if (k < A + Do) v = obs[orow * Do + (k - A)];
        else if (k < A + Do + T) v = (k - A - Do == t) ? 1.f : 0.f;
        else if (k == A + Do + T) v = 1.f;
        ts::split_f16(v, o3[0][j], o3[1][j]);
        ts::split_bf16(v, o3[2][j], o3[3][j]);
    }
#pragma unroll
    for (int pl = 0; pl < 2; ++pl) {
        if (hf.p[0]) *reinterpret_cast<uint4*>(hf.p[pl] + (size_t)r * KP0 + k0) = *reinterpret_cast<const uint4*>(o3[pl]);
        if (hb.p[0]) *reinterpret_cast<uint4*>(hb.p[pl] + (size_t)r * KP0 + k0) = *reinterpret_cast<const uint4*>(o3[2 + pl]);
    }
}
// dst[r][0:ld] = [src[r][0:ncols] | 0..] as two planes (ld a multiple of 8: the padded width NOP); one thread per 8 columns
__global__ void ts_pad64_kernel(const float* __restrict__ src, int N, int ncols, int ld, bf16* __restrict__ hi, bf16* __restrict__ lo) {
    const int g8 = ld / 8;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * g8) return;
    const int r = (int)(i / g8), k0 = (int)(i % g8) * 8;
    __align__(16) bf16 oh[8]; __align__(16) bf16 ol[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) ts::split_bf16(k0 + j < ncols ? src[(size_t)r * ncols + k0 + j] : 0.f, oh[j], ol[j]);
    *reinterpret_cast<uint4*>(hi + (size_t)r * ld + k0) = *reinterpret_cast<const uint4*>(oh);
    *reinterpret_cast<uint4*>(lo + (size_t)r * ld + k0) = *reinterpret_cast<const uint4*>(ol);
}

// the folded output layer (W2 W3, b2 W3 + b3; ActorDerived::w23 / b23) is rebuilt lazily: only forward-only programs read it, updates come in runs
static int ensure_w23(dppo_handle* h, int net, cudaStream_t s) {
    const Geom& g = h->g;
    if (!h->w23_dirty[net] || net == DPPO_NET_CRITIC) return 0;
    const float* w = h->net_w[net]; ActorDerived& d = h->ad[net];
    fold_output_kernel<<<tc_nblk((size_t)(g.H + 1) * g.A, 128), 128, 0, s>>>(w + g.ao.w2, w + g.ao.b2, w + g.ao.w3, w + g.ao.b3, g.H, g.A, d.w23, d.b23);
    TC_KCHECK(h);
    h->w23_dirty[net] = 0;
    return 0;
}
// Folded output layer of one net.  No activation sits between block.l2 and the last Dense (model/common/mlp.py), so
//   out = (a1 W2 + b2 + u) W3 + b3 = [a1 | h0] [W2 W3 ; W0 W3] + ((b2 + b0) W3 + b3),      u = h0 W0 + b0
// with W0 = the h0-order rows of layer 0 ([x | obs | bt[t] | 0..]; the actor's b0 rides in the bt rows, the critic's is `b0`).
// ffold[a][k] (a < NOP, k < H + KP0) = that matrix transposed, as fp16 planes of 2^10 x (f16) or bf16 planes; bfold[a] the bias.
// One thread per (k, a) and one for each bias entry; double accumulation, rounded once.
struct TsFoldArgs {
    const float *w2, *w3, *b2, *b3, *b0;      // [H][H], [H][NO], [H], [NO], [H] or null
    const float *win; int x_rows, x_skip;     // layer-0 rows of h0 columns [0, A): win + k0 * H when k0 < x_rows (else zero)
    int obs_skip;                             // rows of h0 columns [A, A + Do): win + (k0 - A + obs_skip) * H
    const float* bt;                          // rows of h0 columns [A + Do, A + Do + T): bt + (k0 - A - Do) * H, or null
    int A, Do, T, H, NO, KP0, f16;
};
// one warp per output row k (k == H + KP0: the bias row) and 8-column group a0 = 8 blockIdx.y of the output: the lanes split j (16
// products each, fp32), the group's 8 columns of W3 sit transposed and padded in shared memory (conflict-free both ways), the lane
// partials meet in a butterfly.  (A first version accumulated in double: 30 us - the CUDA-core fp64 rate of this part - for sums that
// are rounded to 22-bit planes anyway.  One block per 8 rows for all 64 columns: 20 us on 73 blocks; split by column group the launch
// has 8x the blocks and each stages an eighth of W3.)  gridDim.y = NOP / 8 groups; the groups at and past NO write the zero padding.
__global__ void __launch_bounds__(256) ts_fold_kernel(const TsFoldArgs f, const TsW F, float* __restrict__ bfold, const TsW B23) {
    pdl_grid_begin();
    extern __shared__ float w3t[];               // [8][H + 1]: columns a0 .. a0 + 7 of W3
    const int H = f.H, NO = f.NO, ld = f.H + f.KP0, HP = f.H + 1, a0 = 8 * blockIdx.y;
    const int nq = min(8, NO - a0);              // columns of this group inside the layer (<= 0: the zero padding)
    for (int i0 = threadIdx.x; i0 < H * 8; i0 += blockDim.x * 8) {         // eight loads in flight per thread
        float t8[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) { const int i = i0 + u * blockDim.x; t8[u] = (i < H * 8 && i % 8 < nq) ? __ldg(f.w3 + (size_t)(i / 8) * NO + a0 + i % 8) : 0.f; }
#pragma unroll
        for (int u = 0; u < 8; ++u) { const int i = i0 + u * blockDim.x; if (i < H * 8) w3t[(size_t)(i % 8) * HP + i / 8] = t8[u]; }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k > ld) return;
    const float* row = nullptr; bool bias_row = false;
    if (k < H) row = f.w2 + (size_t)k * H;
    else if (k < ld) {
        const int k0 = k - H;
        if (k0 < f.A) { if (k0 < f.x_rows) row = f.win + (size_t)(k0 + f.x_skip) * H; }
        else if (k0 < f.A + f.Do) row = f.win + (size_t)(k0 - f.A + f.obs_skip) * H;
        else if (k0 < f.A + f.Do + f.T) { if (f.bt) row = f.bt + (size_t)(k0 - f.A - f.Do) * H; }
    } else { row = f.b2; bias_row = true; }
    if (a0 >= NO) row = nullptr;                 // zero columns: nothing to load
    float rv[32];                                // the lane's row elements, all loads in flight at once
#pragma unroll
    for (int q = 0; q < 32; ++q) {
        const int j = lane + 32 * q;
        rv[q] = (row && j < H) ? row[j] : 0.f;
        if (row && bias_row && f.b0 && j < H) rv[q] += f.b0[j];
    }
    {
        float acc[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[q] = 0.f;
        if (row && a0 < NO) {
#pragma unroll
            for (int qq = 0; qq < 32; ++qq) {
                const int j = lane + 32 * qq;
                if (j < H) {
#pragma unroll
                    for (int q = 0; q < 8; ++q) if (a0 + q < NO) acc[q] = fmaf(rv[qq], w3t[(size_t)q * HP + j], acc[q]);
                }
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
#pragma unroll
                for (int q = 0; q < 8; ++q) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], off);
            }
        }
        if (lane < 8) {
            const int a = a0 + lane;
            float v = 0.f;
#pragma unroll
            for (int q = 0; q < 8; ++q) if (q == lane) v = acc[q];
            if (bias_row) bfold[a] = a < NO ? v + f.b3[a] : 0.f;
            else if (f.f16) ts_put_f16(F, (size_t)a * ld + k, v);
            else ts_put(F, (size_t)a * ld + k, v);
            if (!bias_row && k < H) ts_put(B23, (size_t)k * 128 + a, v);          // the backward operand (bf16 planes, row k of W2 W3)
        }
    }
}
static const int TS_MIN_ROWS = 2048;
static bool ts_shapes_ok(const dppo_handle* h) { return h->ts && h->ts->net[0].w1.p[0] != nullptr; }
static bool ts_eligible(const dppo_handle* h, int rows) {
    return h->cfg.precision == DPPO_PREC_BF16X3 && ts_shapes_ok(h) && rows >= TS_MIN_ROWS;
}
static int ts_alloc_w(TsW& w, size_t n) {
    CUDA_TRY(cudaMalloc(&w.p[0], 2 * n * sizeof(bf16)));
    w.p[1] = w.p[0] + n; w.p[2] = nullptr;
    return 0;
}
static bool ts_dw3_fits(const Geom& g);
static int ts_init(dppo_handle* h) {
    if (h->cfg.precision != DPPO_PREC_BF16X3) return 0;
    const Geom& g = h->g;
    TsState* st = new TsState();
    memset(st, 0, sizeof(*st));
    h->ts = st;
    st->KP0 = round_up(g.A + g.Do + g.T + 1, 64);
    // shapes this path does not cover (the widths of the plane GEMMs, the output-layer gradient assembly): stays on FFMA
    if ((g.H % 64) || (g.Hc % 64) || !ts_dw3_fits(g)) return 0;
    for (int net = 0; net < 4; ++net) {
        TsNetW& w = st->net[net];
        const size_t H = net == DPPO_NET_CRITIC ? g.Hc : g.H;
        const size_t NOP = ts_nop(net == DPPO_NET_CRITIC ? 1 : g.A);
        DPPO_TRY(ts_alloc_w(w.w0, st->KP0 * H)); DPPO_TRY(ts_alloc_w(w.w1, H * H));
        DPPO_TRY(ts_alloc_w(w.fw0, st->KP0 * H)); DPPO_TRY(ts_alloc_w(w.fw1, H * H));
        DPPO_TRY(ts_alloc_w(w.ffold, NOP * (H + st->KP0)));
        CUDA_TRY(cudaMalloc(&w.bfold, NOP * sizeof(float)));
        DPPO_TRY(ts_alloc_w(w.w23p, H * 128)); CUDA_TRY(cudaMemset(w.w23p.p[0], 0, 2 * H * 128 * sizeof(bf16)));
        st->fold_dirty[net] = 1;
    }
    return 0;
}
static void ts_destroy(dppo_handle* h) {
    if (!h->ts) return;
    cudaFree(h->ts->dw3_buf);
    for (int net = 0; net < 4; ++net) { TsNetW& w = h->ts->net[net]; cudaFree(w.w0.p[0]); cudaFree(w.w1.p[0]); cudaFree(w.fw0.p[0]); cudaFree(w.fw1.p[0]); cudaFree(w.ffold.p[0]); cudaFree(w.bfold); cudaFree(w.w23p.p[0]); }
    delete h->ts; h->ts = nullptr;
}
// rebuild the plane copies of one net (after set_weights / an optimizer step; the actor's bt table must be current)
static int ts_refresh_net(dppo_handle* h, int net, cudaStream_t s) {
    if (h->cfg.precision != DPPO_PREC_BF16X3 || !ts_shapes_ok(h)) return 0;
    const Geom& g = h->g; const TsNetW& w = h->ts->net[net];
    if (net == DPPO_NET_CRITIC) ts_pack_critic_kernel<<<128, 256, 0, s>>>(h->net_w[net], g.co, g.A, g.Do, g.Hc, h->ts->KP0, w);
    else ts_pack_actor_kernel<<<256, 256, 0, s>>>(h->net_w[net], g.ao, g.A, g.td, g.Do, g.T, g.H, h->ts->KP0, h->ad[net].bt, w);
    TC_KCHECK(h);
    return 0;
}

static int ts_ensure_fold(dppo_handle* h, int net, cudaStream_t s);
// ------------------------------------------------------------------ AdamW and every weight-derived table in one launch
// The optimizer step of [actor_ft | critic] followed by what prep_net rebuilds for both nets (the actor's time tables, the plane
// copies of W1 and of the layer-0 rows), bit-identical to that sequence:
//  * element blocks (after the time blocks): one parameter per thread (adamw_elem); an element of W1 or of a W_in x / obs row also writes its planes.  The
//    zero rows of the layer-0 planes (the critic's x / time rows, the pad rows) never change and are left as prep_net wrote them.
//  * T time blocks (blocks 0 .. T-1): block t evaluates the update of the time MLP, the W_in time rows and b_in itself (from the old w, g,
//    m, v, into shared memory), runs actor_prep_body on those values and writes row A + Do + t of the layer-0 planes (= bt[t]).
//    The last time block to finish (counter) writes those small parameters back; until then every time block still reads the old
//    ones, so the element blocks skip their ranges.
struct TsUpdateArgs {
    float* w; const float* g; float* m; float* v; size_t n, nA;            // [actor_ft | critic] and its optimizer moments
    float lr, alpha, b1, b2, eps, wd; const int *skip0, *skip1;
    ActorOff ao; CriticOff co; int A, td, Do, T, H, Hc, elem_blocks;
    TsNetW wa, wc;                                                           // plane copies of actor_ft / critic
    float *sinemb, *thpre, *temb, *bt; int* done;                            // actor_ft's time tables
};
__device__ __forceinline__ bool ts_update_time_param(const TsUpdateArgs& a, size_t i) {      // written by the last time block
    const size_t wt0 = a.ao.win + (size_t)a.A * a.H, wt1 = wt0 + (size_t)a.td * a.H;
    return i < a.ao.win || (i >= wt0 && i < wt1) || (i >= a.ao.bin && i < a.ao.bin + a.H);
}
__device__ __forceinline__ float ts_update_new(const TsUpdateArgs& a, size_t i, float* mo = nullptr, float* vo = nullptr) {
    float p = a.w[i], mi = a.m[i], vi = a.v[i];
    adamw_elem(p, mi, vi, a.g[i], a.lr, a.alpha, a.b1, a.b2, a.eps, a.wd);
    if (mo) { *mo = mi; *vo = vi; }
    return p;
}
// the parameters the time blocks own, numbered q: [time MLP (q < ao.win, ao.tw1 == 0) | W_in time rows | b_in]
__device__ __forceinline__ size_t ts_update_time_count(const TsUpdateArgs& a) { return a.ao.win + (size_t)(a.td + 1) * a.H; }
__device__ __forceinline__ size_t ts_update_time_index(const TsUpdateArgs& a, size_t q) {
    const size_t nmlp = a.ao.win, ntd = (size_t)a.td * a.H;
    return q < nmlp ? q : (q < nmlp + ntd ? a.ao.win + (size_t)a.A * a.H + (q - nmlp) : a.ao.bin + (q - nmlp - ntd));
}
// the update of every time parameter, eight of them in flight per thread: into sm[q] (WRITE_BACK false) or into w, m, v
template <bool WRITE_BACK>
__device__ __forceinline__ void ts_update_time_params(const TsUpdateArgs& a, float* sm) {
    const size_t nq = ts_update_time_count(a);
    for (size_t q0 = threadIdx.x; q0 < nq; q0 += 8 * (size_t)blockDim.x) {
        float p[8], mi[8], vi[8], gi[8]; size_t idx[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const size_t q = q0 + (size_t)u * blockDim.x;
            idx[u] = q < nq ? ts_update_time_index(a, q) : 0;
            p[u] = a.w[idx[u]]; mi[u] = a.m[idx[u]]; vi[u] = a.v[idx[u]]; gi[u] = a.g[idx[u]];
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const size_t q = q0 + (size_t)u * blockDim.x;
            if (q >= nq) break;
            adamw_elem(p[u], mi[u], vi[u], gi[u], a.lr, a.alpha, a.b1, a.b2, a.eps, a.wd);
            if (WRITE_BACK) { a.w[idx[u]] = p[u]; a.m[idx[u]] = mi[u]; a.v[idx[u]] = vi[u]; }
            else sm[q] = p[u];
        }
    }
}
struct WUpdated {        // actor_prep_body's view of the updated actor: the time parameters staged in shared memory (the only ones it reads)
    const TsUpdateArgs* a; const float* tp;
    __device__ __forceinline__ float operator()(size_t i) const {
        const size_t nmlp = a->ao.win, wt0 = a->ao.win + (size_t)a->A * a->H, ntd = (size_t)a->td * a->H;
        return i < nmlp ? tp[i] : (i < a->ao.bin ? tp[nmlp + (i - wt0)] : tp[nmlp + ntd + (i - a->ao.bin)]);
    }
};
__global__ void __launch_bounds__(512) ts_update_kernel(const TsUpdateArgs a) {
    pdl_grid_begin();
    if ((a.skip0 && *a.skip0) || (a.skip1 && *a.skip1)) return;          // bad minibatch / failed exchange: nothing changes
    const int tid = threadIdx.x;
    if ((int)blockIdx.x >= a.T) {                 // the time blocks come first: their chain is the longest
        const size_t i = (size_t)(blockIdx.x - a.T) * blockDim.x + tid;
        if (i >= a.n || (i < a.nA && ts_update_time_param(a, i))) return;
        float mi, vi;
        const float p = ts_update_new(a, i, &mi, &vi);
        a.w[i] = p; a.m[i] = mi; a.v[i] = vi;
        if (i < a.nA) {
            const size_t H = a.H;
            if (i >= a.ao.w1 && i < a.ao.w1 + H * H) ts_put2(a.wa.w1, a.wa.fw1, i - a.ao.w1, p);
            else if (i >= a.ao.win && i < a.ao.win + (size_t)(a.A + a.td + a.Do) * H) {
                const size_t r = (i - a.ao.win) / H, c = (i - a.ao.win) % H;      // W_in rows [x | time | obs]; h0 order [x | obs | ..]
                ts_put2(a.wa.w0, a.wa.fw0, (r < (size_t)a.A ? r : r - a.td) * H + c, p);
            }
        } else {
            const size_t j = i - a.nA, Hc = a.Hc;
            if (j >= a.co.w1 && j < a.co.w1 + Hc * Hc) ts_put2(a.wc.w1, a.wc.fw1, j - a.co.w1, p);
            else if (j >= a.co.win && j < a.co.win + (size_t)a.Do * Hc) ts_put2(a.wc.w0, a.wc.fw0, (size_t)a.A * Hc + (j - a.co.win), p);
        }
        return;
    }
    const int t = blockIdx.x;
    extern __shared__ float upd_sm[];            // [ts_update_time_count] updated time parameters | actor_prep_body's [4 td]
    ts_update_time_params<false>(a, upd_sm);
    __syncthreads();
    actor_prep_body(t, upd_sm + ts_update_time_count(a), WUpdated{&a, upd_sm}, a.ao, a.A, a.td, a.H, a.sinemb, a.thpre, a.temb, a.bt, nullptr);
    for (int c = tid; c < a.H; c += blockDim.x)  // this thread wrote bt[t][c]
        ts_put2(a.wa.w0, a.wa.fw0, (size_t)(a.A + a.Do + t) * a.H + c, a.bt[(size_t)t * a.H + c]);
    __shared__ int last_flag;
    __threadfence();
    __syncthreads();
    if (tid == 0) last_flag = (atomicAdd(a.done, 1) == a.T - 1) ? 1 : 0;
    __syncthreads();
    if (!last_flag) return;
    ts_update_time_params<true>(a, nullptr);
    if (tid == 0) *a.done = 0;                   // ready for the next launch
}
static size_t ts_update_smem(const Geom& g) { return (g.ao.win + (size_t)(g.td + 1) * g.H + 4 * (size_t)g.td) * sizeof(float); }
static bool ts_update_ok(const dppo_handle* h) {
    return h->cfg.precision == DPPO_PREC_BF16X3 && ts_shapes_ok(h) && 2 * h->g.td <= 512 && h->g.ao.tw1 == 0 && ts_update_smem(h->g) <= 48 * 1024;
}
// AdamW (alpha: the bias-corrected step size of this step) on [actor_ft | critic] with gradient g, then the derived tables of both
// nets: replaces adamw_kernel + prep_net(ACTOR_FT) + prep_net(CRITIC) of the split-precision mode
static int ts_apply_update(dppo_handle* h, cudaStream_t s, const float* g, float lr, float alpha, float wd, const int* skip1) {
    const Geom& gm = h->g; OptState& o = h->opt[DPPO_OPT_FINETUNE]; ActorDerived& d = h->ad[DPPO_NET_ACTOR_FT];
    TsUpdateArgs a;
    a.w = h->net_w[DPPO_NET_ACTOR_FT]; a.g = g; a.m = o.m; a.v = o.v; a.nA = gm.ao.n; a.n = gm.ao.n + gm.co.n;
    a.lr = lr; a.alpha = alpha; a.b1 = h->cfg.adam_beta1; a.b2 = h->cfg.adam_beta2; a.eps = h->cfg.adam_eps; a.wd = wd;
    a.skip0 = h->skip_update; a.skip1 = skip1;
    a.ao = gm.ao; a.co = gm.co; a.A = gm.A; a.td = gm.td; a.Do = gm.Do; a.T = gm.T; a.H = gm.H; a.Hc = gm.Hc;
    a.elem_blocks = tc_nblk(a.n, 512);
    a.wa = h->ts->net[DPPO_NET_ACTOR_FT]; a.wc = h->ts->net[DPPO_NET_CRITIC];
    a.sinemb = d.sinemb; a.thpre = d.thpre; a.temb = d.temb; a.bt = d.bt;
    a.done = reinterpret_cast<int*>(d.dte + (size_t)gm.T * gm.td) + 1;
    CUDA_TRY(launch_pdl(ts_update_kernel, dim3(a.elem_blocks + gm.T), dim3(512), ts_update_smem(gm), s, a)); TC_KCHECK(h);
    mark_weights_changed(h, DPPO_NET_ACTOR_FT); mark_weights_changed(h, DPPO_NET_CRITIC);
    // the folded output layers of the new weights, here rather than lazily at the next update's start: there they ran on the second
    // stream but got SMs only when the actor's persistent L1 drained, and the actor's folded GEMM waited for them
    DPPO_TRY(ts_ensure_fold(h, DPPO_NET_ACTOR_FT, s)); DPPO_TRY(ts_ensure_fold(h, DPPO_NET_CRITIC, s));
    return 0;
}

// ------------------------------------------------------------------ one residual MLP on N rows, every tensor as planes
// The output layer is folded: out = [a1 | h0] [W2 W3 ; W0 W3] + bfold, so block.l2's H x H product is skipped and v never formed (the
// caller has run ts_ensure_fold).  The weight gradient of the output layer is assembled from a1^T dout and h0^T dout (ts_dw3_assemble_kernel).
struct TsMlp {
    const TsNetW* W; int H, NO, NOP, act1, KP0, net, din;
    int fp;                                // FORWARD GEMMs: 4 = two fp16 planes + two accumulators (22 bits) when the net has kinks behind it,
                                           // 2 = two bf16 planes, one accumulator (16 bits).  h0 / a0 / a1 carry that format.
    const float *b0, *b1;
    SplitT h0, a0, a1, g0, g1, dh1, du;    // g0 / g1: Mish gates mish'(pre-activation) of layer 0 / block.l1 (two planes)
    SplitT h0b, a0b, a1b;                  // fp = 4 with a backward pass: bf16 copies (two planes) for the weight-gradient GEMMs
    cudaEvent_t fold_ev;                   // when set: the folded operands are being rebuilt on another stream; wait in front of the folded GEMM
    uint32_t *m0, *m1;                     // ReLU bit masks [N][H/32] of layer 0 / block.l1
    float* out;                            // [N][NO] fp32
};
// rebuild the folded output layer of one net if its weights changed (lazily: set_weights / AdamW only mark it stale)
static int ts_ensure_fold(dppo_handle* h, int net, cudaStream_t s) {
    if (!h->ts->fold_dirty[net]) return 0;
    const Geom& g = h->g; const TsNetW& W = h->ts->net[net]; const float* w = h->net_w[net];
    TsFoldArgs f; memset(&f, 0, sizeof(f));
    f.A = g.A; f.Do = g.Do; f.T = g.T; f.KP0 = h->ts->KP0;
    if (net == DPPO_NET_CRITIC) {
        f.H = g.Hc; f.NO = 1; f.w2 = w + g.co.w2; f.w3 = w + g.co.w3; f.b2 = w + g.co.b2; f.b3 = w + g.co.b3; f.b0 = w + g.co.bin;
        f.win = w + g.co.win; f.x_rows = 0; f.obs_skip = 0; f.bt = nullptr;
        f.f16 = h->cfg.critic_act == DPPO_ACT_RELU ? 1 : 0;
    } else {
        f.H = g.H; f.NO = g.A; f.w2 = w + g.ao.w2; f.w3 = w + g.ao.w3; f.b2 = w + g.ao.b2; f.b3 = w + g.ao.b3; f.b0 = nullptr;
        f.win = w + g.ao.win; f.x_rows = g.A; f.x_skip = 0; f.obs_skip = g.A + g.td; f.bt = h->ad[net].bt;
        f.f16 = 1;
    }
    static bool attr_set_dev[64] = {};
    if (!attr_set_dev[h->device & 63]) { CUDA_TRY(cudaFuncSetAttribute(ts_fold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024)); attr_set_dev[h->device & 63] = true; }
    const size_t sm = (size_t)(f.H + 1) * 8 * sizeof(float);
    if (sm > 96 * 1024 || f.H > 1024 || f.NO > 128) DPPO_FAIL(-7, "ts_ensure_fold: output layer too wide for the fold kernel");
    CUDA_TRY(launch_pdl(ts_fold_kernel, dim3(tc_nblk((size_t)(f.H + f.KP0 + 1), 8), ts_nop(f.NO) / 8), dim3(256), sm, s, f, W.ffold, W.bfold, W.w23p));
    TC_KCHECK(h);
    h->ts->fold_dirty[net] = 0;
    return 0;
}
static void ts_actor_mlp(const dppo_handle* h, int net, TsMlp& m) {
    const Geom& g = h->g; const float* w = h->net_w[net];
    memset(&m, 0, sizeof(m));
    m.W = &h->ts->net[net]; m.H = g.H; m.NO = g.A; m.NOP = ts_nop(g.A); m.act1 = h->cfg.actor_act + 1; m.KP0 = h->ts->KP0; m.net = net; m.din = g.Din;
    m.fp = 4;                                                                        // ReLU kinks and the +-1 clip of x0 behind eps
    m.b0 = nullptr; m.b1 = w + g.ao.b1;                                              // b_in rides in W0's one-hot rows (bt table)
}
static void ts_critic_mlp(const dppo_handle* h, TsMlp& m) {
    const Geom& g = h->g; const float* w = h->net_w[DPPO_NET_CRITIC];
    memset(&m, 0, sizeof(m));
    m.W = &h->ts->net[DPPO_NET_CRITIC]; m.H = g.Hc; m.NO = 1; m.NOP = ts_nop(1); m.act1 = h->cfg.critic_act + 1; m.KP0 = h->ts->KP0; m.net = DPPO_NET_CRITIC; m.din = g.Do;
    m.fp = h->cfg.critic_act == DPPO_ACT_RELU ? 4 : 2;                               // Mish is smooth
    m.b0 = w + g.co.bin; m.b1 = w + g.co.b1;
}
static SplitT ts_take(dppo_handle* h, size_t n, int planes) {
    SplitT t = split_null();
    for (int pl = 0; pl < planes; ++pl) t.p[pl] = ws_take<bf16>(h, n);
    return t;
}
// own_h0 = false: the net reads another net's input planes (h0, h0b), which the caller points it at
static void ts_mlp_take(dppo_handle* h, int N, TsMlp& m, bool bwd, bool own_h0 = true) {
    const size_t n = (size_t)N * m.H;
    if (own_h0) m.h0 = ts_take(h, (size_t)N * m.KP0, 2);
    m.a0 = ts_take(h, n, 2); m.a1 = ts_take(h, n, 2);
    if (m.act1 == 2) { m.g0 = ts_take(h, n, 2); m.g1 = ts_take(h, n, 2); }
    if (bwd) { m.dh1 = ts_take(h, n, 2); m.du = ts_take(h, n, 2); }
    if (bwd && m.fp == 4) { if (own_h0) m.h0b = ts_take(h, (size_t)N * m.KP0, 2); m.a0b = ts_take(h, n, 2); m.a1b = ts_take(h, n, 2); }
    m.m0 = ws_take<uint32_t>(h, (size_t)N * (m.H / 32)); m.m1 = ws_take<uint32_t>(h, (size_t)N * (m.H / 32));
}
static ts::Operand ts_op(const bf16* const* p, size_t off, bool mn_major, int64_t mn, int64_t k, int64_t ld) {
    ts::Operand o; o.mn_major = mn_major; o.mn = mn; o.k = k; o.ld = ld;
    for (int pl = 0; pl < ts::MAXP; ++pl) o.p[pl] = p[pl] ? p[pl] + off : nullptr;
    return o;
}
static ts::Operand tsK(const SplitT& t, int64_t mn, int64_t k, int64_t ld) { return ts_op(t.p, 0, false, mn, k, ld); }
static ts::Operand tswK(const TsW& w, size_t off, int64_t mn, int64_t k, int64_t ld) { return ts_op(w.p, off, false, mn, k, ld); }
static ts::Operand tswMN(const TsW& w, size_t off, int64_t mn, int64_t k, int64_t ld) { return ts_op(w.p, off, true, mn, k, ld); }
static ts::Gemm ts_gemm_of(ts::Operand A, ts::Operand B, int M, int N, int planes, int dual = 0) {
    ts::Gemm g; memset(&g, 0, sizeof(g));
    g.A = A; g.B = B; g.M = M; g.N = N; g.splits = 1; g.planes = planes; g.dual = dual; g.epi.M = M; g.epi.N = N;
    return g;
}
static int ts_run(dppo_handle* h, cudaStream_t s, const ts::Gemm& g) { const int r = ts::launch(h, s, g); return r < 0 ? r : 0; }
// a layer on the pair kernel: out (planes) = epilogue(A B)
static tsp::Gemm tsp_gemm_of(ts::Operand A, ts::Operand B, int M, int N, int planes, const SplitT& out, int out_planes, int ld_out) {
    tsp::Gemm g; memset(&g, 0, sizeof(g));
    if (planes == 4) { planes = 2; out_planes = 2; g.f16 = 1; g.dual = 1; g.epi.scale = 1.0f / ts::F16_WSCALE; }   // fp16 planes in and out
    else g.dual = planes == 3 ? 1 : 0;
    g.A = A; g.B = B; g.M = M; g.N = N; g.planes = planes;
    for (int pl = 0; pl < ts::MAXP; ++pl) g.out[pl] = out.p[pl];
    g.ld_out = ld_out; g.epi.M = M; g.epi.N = N; g.epi.out_planes = out_planes;
    return g;
}

// phase 0: the whole forward; 1: L0 and L1 only; 2: what follows L1 (lets a caller enqueue other streams' work in between)
static int ts_mlp_forward(dppo_handle* h, cudaStream_t s, const TsMlp& m, int N, int phase = 0) {
    const int H = m.H, KP0 = m.KP0, P = m.fp; const TsNetW& W = *m.W;
    const bool f16 = P == 4;
    const TsW& Ww0 = f16 ? W.fw0 : W.w0; const TsW& Ww1 = f16 ? W.fw1 : W.w1;
    tsp::Gemm g;
    if (phase != 2) {
    // L0: a0 = act(h0 W0 (+ b0))
    g = tsp_gemm_of(tsK(m.h0, N, KP0, KP0), tswMN(Ww0, 0, H, KP0, H), N, H, P, m.a0, P, H);
    g.epi.bias = m.b0; g.epi.act = m.act1;
    if (m.a0b.p[0]) { g.out2[0] = m.a0b.p[0]; g.out2[1] = m.a0b.p[1]; g.epi.out2 = 1; }
    if (m.act1 == 1) { g.epi.mask_out = m.m0; g.epi.ldm = H / 32; } else if (m.act1 == 2) { g.epi.gate_out = 1; g.gate[0] = m.g0.p[0]; g.gate[1] = m.g0.p[1]; }
    g.alg_flops = 2.0 * N * (double)m.din * H;
    DPPO_TRY(tsp::launch(h, s, g));
    // L1: a1 = act(a0 W1 + b1)
    g = tsp_gemm_of(tsK(m.a0, N, H, H), tswMN(Ww1, 0, H, H, H), N, H, P, m.a1, P, H);
    g.epi.bias = m.b1; g.epi.act = m.act1;
    if (m.a1b.p[0]) { g.out2[0] = m.a1b.p[0]; g.out2[1] = m.a1b.p[1]; g.epi.out2 = 1; }
    if (m.act1 == 1) { g.epi.mask_out = m.m1; g.epi.ldm = H / 32; } else if (m.act1 == 2) { g.epi.gate_out = 1; g.gate[0] = m.g1.p[0]; g.gate[1] = m.g1.p[1]; }
    DPPO_TRY(tsp::launch(h, s, g));
    }
    if (phase == 1) return 0;
    // no activation between block.l2 and the output layer: out = [a1 | h0] [W2 W3 ; W0 W3] + bfold, one narrow GEMM
    const int nb = m.NO <= 32 ? 32 : m.NOP;                              // ffold rows the GEMM reads (the B box)
    ts::Gemm o = ts_gemm_of(tsK(m.a1, N, H, H), tswK(W.ffold, 0, nb, H, H + KP0), N, m.NO, 2, f16 ? 1 : 0);
    o.A2 = tsK(m.h0, N, KP0, KP0); o.B2 = tswK(W.ffold, (size_t)H, nb, KP0, H + KP0);
    if (f16) { o.f16 = 1; o.epi.scale = 1.0f / ts::F16_WSCALE; }
    o.epi.bias = W.bfold; o.epi.out_f32 = m.out; o.epi.ld_f32 = m.NO;
    o.alg_flops = 2.0 * N * ((double)H * H + (double)H * m.NO);        // the algorithmic work it stands for
    if (m.fold_ev) CUDA_TRY(cudaStreamWaitEvent(s, m.fold_ev, 0));
    DPPO_TRY(ts_run(h, s, o));
    return 0;
}
// backward chain of the residual MLP from dout [N][NOP] (two planes, zero padded): dh1 = (dout (W2 W3)^T) . act'(h1),
// du = (dh1 W1^T) . act'(u).  dv = dout W3^T has rank NO and is never formed: dh1 is ONE K = NOP product, and everything else dv
// fed - dW2 = a1^T dv = (a1^T dout) W3^T, the residual part of dW0 = (h0^T dout) W3^T, db2 = (1^T dout) W3^T - is assembled from the small
// products a1^T dout / h0^T dout the folded output layer needs anyway (ts_dw3_assemble_kernel).
// cpart [ceil(N/32)][2][H]: per 32-row block column sums of dh1 (slot 1 = db1), written by the epilogue; slot 0 stays unwritten.
static int ts_mlp_backward_dx(dppo_handle* h, cudaStream_t s, const TsMlp& m, const SplitT& dout, int N, float* cpart) {
    const int H = m.H; const TsNetW& W = *m.W;
    tsp::Gemm g = tsp_gemm_of(tsK(dout, N, m.NOP, m.NOP), tswK(W.w23p, 0, H, m.NOP, 128), N, H, 2, m.dh1, 2, H);
    g.alg_flops = 2.0 * N * ((double)m.NO * H + (double)H * H);                  // the two products it stands for
    g.epi.colsum_part = cpart + H; g.epi.colsum_ld = 2 * H;
    if (m.act1 == 1) { g.epi.mask_in = m.m1; g.epi.ldm = H / 32; } else if (m.act1 == 2) { g.epi.gate_in[0] = m.g1.p[0]; g.epi.gate_in[1] = m.g1.p[1]; g.epi.ldg = H; }
    DPPO_TRY(tsp::launch(h, s, g));
    g = tsp_gemm_of(tsK(m.dh1, N, H, H), tswK(W.w1, 0, H, H, H), N, H, 2, m.du, 2, H);
    if (m.act1 == 1) { g.epi.mask_in = m.m0; g.epi.ldm = H / 32; } else if (m.act1 == 2) { g.epi.gate_in[0] = m.g0.p[0]; g.epi.gate_in[1] = m.g0.p[1]; g.epi.ldg = H; }
    DPPO_TRY(tsp::launch(h, s, g));
    return 0;
}
// the four weight-gradient products of one net for the grouped pair kernel: dW1 = a0^T dh1, the layer-0 product handed over as du^T h0
// (wide operand on M, output written transposed into dw0 [KP0][H]), g1 = a1^T dout [H][NO] and g0 = h0^T dout [KP0][NO]; dW2, dW3 and
// the residual part of dW0 come out of g1 / g0 (see ts_mlp_backward_dx).  Returns the number of problems.
static int ts_mlp_dw_descs(const TsMlp& m, const SplitT& dout, int N, float* gnet, size_t ow1, float* dw0, tsp::DwDesc* d, float* g1, float* g0) {
    const int H = m.H, KP0 = m.KP0; const double r = (double)N; const SplitT none = split_null();
    // (fp = 4: the bf16 copies of the activations - one tcgen05.mma cannot take an fp16 and a bf16 operand, and the gradients are bf16)
    const bool f = m.fp == 4;
    const SplitT& a0 = f ? m.a0b : m.a0; const SplitT& a1 = f ? m.a1b : m.a1; const SplitT& h0 = f ? m.h0b : m.h0;
    d[0] = tsp::DwDesc{a0, H, m.dh1, H, none, none, gnet + ow1, H, H, H, 0, 2.0 * r * H * H};
    d[1] = tsp::DwDesc{m.du, H, h0, KP0, none, none, dw0, H, KP0, H, 1, 2.0 * r * m.din * H};
    d[2] = tsp::DwDesc{a1, H, dout, m.NOP, none, none, g1, H, m.NO, m.NO, 0, 2.0 * r * (H * m.NO + (double)H * H)};
    d[3] = tsp::DwDesc{h0, KP0, dout, m.NOP, none, none, g0, KP0, m.NO, m.NO, 0, 0.0};
    return 4;
}
// dW3[j][a] = sum_r v[r][j] dout[r][a] with v = a1 W2 + (b2 + b0) + h0 W0 never formed:
//   dW3 = W2^T (a1^T dout) + W0^T (h0^T dout) + (b2 + b0) (1^T dout),   1^T dout = the row of h0^T dout that belongs to h0's ones column
// g1 = a1^T dout [H][NO], g0 = h0^T dout [KP0][NO] come from the grouped weight-gradient launch.  One thread per (a, j), j fastest.
struct TsDw3Args {
    const float *w2, *b2, *b0, *win, *bt, *g1, *g0; float* out;
    int x_rows, x_skip, obs_skip, A, Do, T, H, NO, KP0;
    // what dv = dout W3^T would have fed, from the same two small products (rank NO):
    //   dW2 = g1 W3^T [H][H],   dw0 [KP0][H] += g0 W3^T (the residual path's share of the layer-0 gradient),   db2 = (1^T dout) W3^T
    const float* w3; float *dw2, *dw0, *db2;
};
// Grid = (32-column chunk of j) x (KS slices of k): a block sums its k slice for its 32 columns (lane = j: every W2 / W0 read is a
// coalesced 128-byte row segment, all of a warp's loads in flight at once; g1 / g0 rows in shared memory), writes the partial
// [32][NO] tile, and the LAST block of a column chunk to finish (a counter per chunk) adds the KS partials in slice order - the result
// does not depend on which block that is.  (A first version walked all k in one block per chunk: 41 us of serialised load latency.)
// WIDE (NO > 32): the warp partials pass through shared memory DW3_WC columns at a time ([16][32][DW3_WC] instead of [16][32][NO]);
// every output keeps the same sums in the same order.
constexpr int DW3_KS = 8, DW3_WC = 16;
template <bool WIDE>
__device__ __forceinline__ void ts_dw3_assemble_body(const TsDw3Args& f, int bid, float* sm, float* __restrict__ part, int* __restrict__ done) {
    const int H = f.H, NO = f.NO, KT = f.A + f.Do + f.T, K = H + KT;       // k < H: W2 rows; then the h0-order rows of layer 0
    const int jc = bid / DW3_KS, ks = bid % DW3_KS;
    const int kper = (K + DW3_KS - 1) / DW3_KS, kbeg = ks * kper, kend = min(K, kbeg + kper);
    const int NC = WIDE ? DW3_WC : NO;                // columns per pass
    float* gs = sm;                                   // [kper][NO]
    float* red = gs + (size_t)kper * NO;              // [16][32][NC]
    __shared__ int last_flag;
    for (int i = threadIdx.x; i < (kend - kbeg) * NO; i += blockDim.x) {
        const int k = kbeg + i / NO, a = i % NO;
        gs[i] = k < H ? f.g1[(size_t)k * NO + a] : f.g0[(size_t)(k - H) * NO + a];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5, j = jc * 32 + lane;
    auto row_of = [&](int k) -> const float* {
        if (k < H) return f.w2 + (size_t)k * H;
        const int k0 = k - H;
        if (k0 < f.A) return k0 < f.x_rows ? f.win + (size_t)(k0 + f.x_skip) * H : nullptr;
        if (k0 < f.A + f.Do) return f.win + (size_t)(k0 - f.A + f.obs_skip) * H;
        return f.bt ? f.bt + (size_t)(k0 - f.A - f.Do) * H : nullptr;
    };
    float wv[8];                                      // this warp's k: kbeg + warp + u * nw (kper <= 8 * nw)
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const int k = kbeg + warp + u * nw;
        const float* row = (k < kend && j < H) ? row_of(k) : nullptr;
        wv[u] = row ? row[j] : 0.f;
    }
    float* mine = part + ((size_t)jc * DW3_KS + ks) * 32 * NO;
    for (int c0 = 0; c0 < NO; c0 += NC) {
        const int nc = min(NC, NO - c0);
        for (int a = 0; a < nc; ++a) {
            float acc = 0.f;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int kl = warp + u * nw;
                if (kbeg + kl < kend) acc = fmaf(wv[u], gs[(size_t)kl * NO + c0 + a], acc);
            }
            red[((size_t)warp * 32 + lane) * nc + a] = acc;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < 32 * nc; i += blockDim.x) {
            float s = 0.f;
            for (int w = 0; w < nw; ++w) s += red[(size_t)w * 32 * nc + i];
            mine[(size_t)(i / nc) * NO + c0 + i % nc] = s;
        }
        if (WIDE) __syncthreads();                    // red is overwritten by the next pass
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last_flag = (atomicAdd(done + jc, 1) == DW3_KS - 1) ? 1 : 0;
    __syncthreads();
    if (!last_flag) return;
    __threadfence();
    const float* ones = f.g0 + (size_t)KT * NO;        // g0 row A + Do + T = 1^T dout
    for (int i = threadIdx.x; i < 32 * NO; i += blockDim.x) {
        const int l = i / NO, a = i % NO, jj = jc * 32 + l;
        if (jj >= H) continue;
        float s = 0.f;
        for (int q = 0; q < DW3_KS; ++q) s += __ldcg(part + ((size_t)jc * DW3_KS + q) * 32 * NO + i);
        const float bias = f.b2[jj] + (f.b0 ? f.b0[jj] : 0.f);
        f.out[(size_t)jj * NO + a] = fmaf(bias, ones[a], s);
    }
    if (threadIdx.x == 0) done[jc] = 0;                // ready for the next launch
}
// rows q of [g1 ; g0 ; 1^T dout] times W3^T: a block takes DW3_RB rows, thread j keeps row j of W3 in registers
constexpr int DW3_RB = 8;
__device__ __forceinline__ void ts_rank_rows_body(const TsDw3Args& f, int bid, float* sm, int row_begin, int row_end) {
    const int H = f.H, NO = f.NO, nrows = min(H + f.KP0 + 1, row_end), q0 = row_begin + bid * DW3_RB;
    const int ones = f.A + f.Do + f.T;
    for (int i = threadIdx.x; i < DW3_RB * NO; i += blockDim.x) {
        const int q = q0 + i / NO, a = i % NO;
        float v = 0.f;
        if (q < H) v = f.g1[(size_t)q * NO + a];
        else if (q < H + f.KP0) v = f.g0[(size_t)(q - H) * NO + a];
        else if (q == H + f.KP0) v = f.g0[(size_t)ones * NO + a];
        sm[i] = v;
    }
    // W3 through shared memory: coalesced, eight loads in flight per thread (a thread fetching its own row straight from global memory -
    // 24 strided scalar loads - made the 65-row first phase a 16 us kernel)
    float* w3s = sm + DW3_RB * NO;              // [H][NO + 1]
    const int n3 = H * NO;
    for (int i0 = threadIdx.x; i0 < n3; i0 += blockDim.x * 8) {
        float t8[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) { const int i = i0 + u * blockDim.x; t8[u] = i < n3 ? __ldg(f.w3 + i) : 0.f; }
#pragma unroll
        for (int u = 0; u < 8; ++u) { const int i = i0 + u * blockDim.x; if (i < n3) w3s[(i / NO) * (NO + 1) + i % NO] = t8[u]; }
    }
    __syncthreads();
    for (int j = threadIdx.x; j < H; j += blockDim.x) {
        float w3r[32];
#pragma unroll
        for (int a = 0; a < 32; ++a) w3r[a] = a < NO ? w3s[j * (NO + 1) + a] : 0.f;
        float old[DW3_RB];                           // the dw0 entries this thread adds to, all eight loads in flight
#pragma unroll
        for (int r = 0; r < DW3_RB; ++r) {
            const int q = q0 + r;
            old[r] = (q >= H && q < H + f.KP0 && q < nrows) ? f.dw0[(size_t)(q - H) * H + j] : 0.f;
        }
#pragma unroll
        for (int r = 0; r < DW3_RB; ++r) {
            const int q = q0 + r;
            if (q >= nrows) break;
            float acc = 0.f;
#pragma unroll
            for (int a = 0; a < 32; ++a) if (a < NO) acc = fmaf(sm[r * NO + a], w3r[a], acc);
            if (q < H) f.dw2[(size_t)q * H + j] = acc;
            else if (q < H + f.KP0) f.dw0[(size_t)(q - H) * H + j] = old[r] + acc;
            else f.db2[j] = acc;
        }
    }
}
// The same rows for 32 < NO <= 128: W3 passes through shared memory 32 columns at a time ([H][33]); a thread's eight sums run on across the
// passes, so each is the same a = 0 .. NO - 1 chain as above.
__device__ __forceinline__ void ts_rank_rows_wide_body(const TsDw3Args& f, int bid, float* sm, int row_begin, int row_end) {
    const int H = f.H, NO = f.NO, nrows = min(H + f.KP0 + 1, row_end), q0 = row_begin + bid * DW3_RB;
    const int ones = f.A + f.Do + f.T;
    for (int i = threadIdx.x; i < DW3_RB * NO; i += blockDim.x) {
        const int q = q0 + i / NO, a = i % NO;
        float v = 0.f;
        if (q < H) v = f.g1[(size_t)q * NO + a];
        else if (q < H + f.KP0) v = f.g0[(size_t)(q - H) * NO + a];
        else if (q == H + f.KP0) v = f.g0[(size_t)ones * NO + a];
        sm[i] = v;
    }
    float* w3s = sm + DW3_RB * NO;                   // [H][33]: columns [c0, c0 + 32) of W3
    for (int j0 = 0; j0 < H; j0 += blockDim.x) {     // the same trip count in every thread: the passes below synchronise the block
        const int j = j0 + (int)threadIdx.x;
        float old[DW3_RB], acc[DW3_RB];
#pragma unroll
        for (int r = 0; r < DW3_RB; ++r) {
            const int q = q0 + r;
            old[r] = (j < H && q >= H && q < H + f.KP0 && q < nrows) ? f.dw0[(size_t)(q - H) * H + j] : 0.f;
            acc[r] = 0.f;
        }
        for (int c0 = 0; c0 < NO; c0 += 32) {
            const int nc = min(32, NO - c0), n3 = H * nc;
            __syncthreads();                          // the previous pass has read w3s (and, first time, sm is complete)
            for (int i0 = threadIdx.x; i0 < n3; i0 += blockDim.x * 8) {
                float t8[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) { const int i = i0 + u * blockDim.x; t8[u] = i < n3 ? __ldg(f.w3 + (size_t)(i / nc) * NO + c0 + i % nc) : 0.f; }
#pragma unroll
                for (int u = 0; u < 8; ++u) { const int i = i0 + u * blockDim.x; if (i < n3) w3s[(i / nc) * 33 + i % nc] = t8[u]; }
            }
            __syncthreads();
            if (j < H) {
                float w3r[32];
#pragma unroll
                for (int a = 0; a < 32; ++a) w3r[a] = a < nc ? w3s[j * 33 + a] : 0.f;
#pragma unroll
                for (int r = 0; r < DW3_RB; ++r) {
#pragma unroll
                    for (int a = 0; a < 32; ++a) if (a < nc) acc[r] = fmaf(sm[r * NO + c0 + a], w3r[a], acc[r]);
                }
            }
        }
        if (j >= H) continue;
#pragma unroll
        for (int r = 0; r < DW3_RB; ++r) {
            const int q = q0 + r;
            if (q >= nrows) break;
            if (q < H) f.dw2[(size_t)q * H + j] = acc[r];
            else if (q < H + f.KP0) f.dw0[(size_t)(q - H) * H + j] = old[r] + acc[r];
            else f.db2[j] = acc[r];
        }
    }
}
// phase 0: the rows that feed dw0 and db2 (q >= H; the tail kernel reads dw0, so these run first, on the main stream); phase 1: dW3 and the
// dW2 rows (q < H), which nothing but AdamW reads - next to the tail kernel on the second stream.  WIDE: the actor has 32 < NO <= 128 outputs
// (the critic's one output always takes the narrow bodies).
template <bool WIDE>
__global__ void __launch_bounds__(512) ts_dw3_assemble_kernel(const TsDw3Args fa, int blocks_a, const TsDw3Args fc, int blocks_c,
                                                              float* __restrict__ part, int* __restrict__ done, int rank_a, int rank_c, int phase) {
    pdl_grid_begin();
    extern __shared__ float dw3_sm[];
    int b = blockIdx.x;
    if (phase == 1) {
        if (b < blocks_a) { ts_dw3_assemble_body<WIDE>(fa, b, dw3_sm, part, done); return; }
        b -= blocks_a;
        if (b < blocks_c) { ts_dw3_assemble_body<false>(fc, b, dw3_sm, part + (size_t)blocks_a * 32 * fa.NO, done + blocks_a / DW3_KS); return; }
        b -= blocks_c;
    }
    const int ra0 = phase == 0 ? fa.H : 0, ra1 = phase == 0 ? fa.H + fa.KP0 + 1 : fa.H;
    const int rc0 = phase == 0 ? fc.H : 0, rc1 = phase == 0 ? fc.H + fc.KP0 + 1 : fc.H;
    if (b < rank_a) {
        if (WIDE) ts_rank_rows_wide_body(fa, b, dw3_sm, ra0, ra1); else ts_rank_rows_body(fa, b, dw3_sm, ra0, ra1);
        return;
    }
    b -= rank_a;
    if (b < rank_c) ts_rank_rows_body(fc, b, dw3_sm, rc0, rc1);
}
static inline int tsDW3KS() { return DW3_KS; }
// the assembly's k slice of one net (rows of [W2 ; layer-0 rows] per block) and its dynamic shared memory: the larger of the dW3 body's
// [kper][NO] + [16][32][NC] and the rank-rows body's [DW3_RB][NO] + [H][N3 + 1] (WIDE, NO > 32: NC = DW3_WC, N3 = 32)
static int ts_dw3_kper(const Geom& g, int H) { return (H + g.A + g.Do + g.T + DW3_KS - 1) / DW3_KS; }
static size_t ts_dw3_net_smem(const Geom& g, int H, int NO) {
    const bool w = NO > 32;
    const int nc = w ? DW3_WC : NO, n3 = w ? 32 : NO;
    const size_t a = (size_t)ts_dw3_kper(g, H) * NO + 16 * 32 * nc, b = (size_t)DW3_RB * NO + (size_t)H * (n3 + 1);
    return (a > b ? a : b) * sizeof(float);
}
static size_t ts_dw3_smem(const Geom& g) {
    const size_t a = ts_dw3_net_smem(g, g.H, g.A), c = ts_dw3_net_smem(g, g.Hc, 1);
    return a > c ? a : c;
}
// the shapes the assembly covers, for ts_init (a handle outside them runs this mode on FFMA) and the launch: a block's 16 warps hold
// at most 8 k rows each, shared memory up to 100 KB.  (The 256 chunk counters cover any accepted width: H, Hc <= 1024.)
static bool ts_dw3_fits(const Geom& g) {
    return g.A <= 128 && ts_dw3_kper(g, g.H) <= 128 && ts_dw3_kper(g, g.Hc) <= 128 && ts_dw3_smem(g) <= 100 * 1024;
}
// gnet: this net's slice of the flat gradient; dw0: its [KP0][H] layer-0 staging buffer
static TsDw3Args ts_dw3_args(const dppo_handle* h, int net, const float* g1, const float* g0, float* gnet, float* dw0) {
    const Geom& g = h->g; const float* w = h->net_w[net];
    TsDw3Args f; memset(&f, 0, sizeof(f));
    f.A = g.A; f.Do = g.Do; f.T = g.T; f.KP0 = h->ts->KP0; f.g1 = g1; f.g0 = g0; f.dw0 = dw0;
    if (net == DPPO_NET_CRITIC) {
        f.H = g.Hc; f.NO = 1; f.w2 = w + g.co.w2; f.b2 = w + g.co.b2; f.b0 = w + g.co.bin; f.win = w + g.co.win; f.x_rows = 0; f.obs_skip = 0; f.bt = nullptr;
        f.w3 = w + g.co.w3; f.out = gnet + g.co.w3; f.dw2 = gnet + g.co.w2; f.db2 = gnet + g.co.b2;
    } else {
        f.H = g.H; f.NO = g.A; f.w2 = w + g.ao.w2; f.b2 = w + g.ao.b2; f.b0 = nullptr; f.win = w + g.ao.win; f.x_rows = g.A; f.x_skip = 0;
        f.obs_skip = g.A + g.td; f.bt = h->ad[net].bt;
        f.w3 = w + g.ao.w3; f.out = gnet + g.ao.w3; f.dw2 = gnet + g.ao.w2; f.db2 = gnet + g.ao.b2;
    }
    return f;
}
// launches the assembly for the actor (and the critic when gc1 != nullptr): dW3, dW2, db2 and the residual share of dw0.  Must run after the
// grouped weight-gradient launch (g1, g0, dw0) and BEFORE anything that reads dw0 (the tail kernel)
// phase 0 / 1: see the kernel; phase -1: both, one after the other on s
static int ts_dw3_assemble(dppo_handle* h, cudaStream_t s, int actor_net, const float* ga1, const float* ga0, float* gneta, float* dw0a,
                           const float* gc1, const float* gc0, float* gnetc, float* dw0c, int phase = -1) {
    if (phase < 0) {
        DPPO_TRY(ts_dw3_assemble(h, s, actor_net, ga1, ga0, gneta, dw0a, gc1, gc0, gnetc, dw0c, 0));
        return ts_dw3_assemble(h, s, actor_net, ga1, ga0, gneta, dw0a, gc1, gc0, gnetc, dw0c, 1);
    }
    const Geom& g = h->g;
    const TsDw3Args fa = ts_dw3_args(h, actor_net, ga1, ga0, gneta, dw0a);
    TsDw3Args fc = fa; int nbc = 0, nrc = 0;
    const int KP0r = h->ts->KP0 + 1;
    const int nra = phase == 0 ? tc_nblk((size_t)KP0r, DW3_RB) : tc_nblk((size_t)g.H, DW3_RB);
    if (gc1) {
        fc = ts_dw3_args(h, DPPO_NET_CRITIC, gc1, gc0, gnetc, dw0c); nbc = tc_nblk((size_t)g.Hc, 32) * tsDW3KS();
        nrc = phase == 0 ? tc_nblk((size_t)KP0r, DW3_RB) : tc_nblk((size_t)g.Hc, DW3_RB);
    }
    const int nba = tc_nblk((size_t)g.H, 32) * tsDW3KS();
    const bool wide = fa.NO > 32;
    // (sized for both nets also when the critic is absent)
    const size_t sm = ts_dw3_smem(g);
    auto kern = wide ? ts_dw3_assemble_kernel<true> : ts_dw3_assemble_kernel<false>;
    static bool attr_set_dev[2][64] = {};
    if (!attr_set_dev[wide][h->device & 63]) { CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024)); attr_set_dev[wide][h->device & 63] = true; }
    if (!ts_dw3_fits(g)) DPPO_FAIL(-7, "ts_dw3_assemble: shape not covered (ts_init routes it to FFMA)");
    TsState* st = h->ts;
    // buffer: [256 chunk counters (always at the front: launches with and without the critic share them, every launch leaves them zero)
    //          | partial tiles]
    const size_t need = 1024 + ((size_t)nba * 32 * g.A + (size_t)nbc * 32) * sizeof(float);
    if (st->dw3_bytes < need) {
        CUDA_TRY(cudaStreamSynchronize(s));
        if (st->dw3_buf) cudaFree(st->dw3_buf);
        CUDA_TRY(cudaMalloc(&st->dw3_buf, need)); CUDA_TRY(cudaMemsetAsync(st->dw3_buf, 0, need, s));
        st->dw3_bytes = need;
    }
    int* done = reinterpret_cast<int*>(st->dw3_buf);
    float* partb = reinterpret_cast<float*>(st->dw3_buf + 1024);
    CUDA_TRY(launch_pdl(kern, dim3((phase == 1 ? nba + nbc : 0) + nra + nrc), dim3(512), sm, s, fa, nba, fc, nbc, partb, done, nra, nrc, phase));
    TC_KCHECK(h);
    return 0;
}
static size_t ts_part_floats(const dppo_handle* h, int H) {
    const size_t a = tc_part_floats(h, H), b = (size_t)(h->sm_count / 2 + 1) * 65536;
    return a > b ? a : b;
}
// ------------------------------------------------------------------ forward-only programs
// the buffers ts_actor_forward appends for N rows
static void ts_actor_forward_take(dppo_handle* h, int net, int N, TsMlp& m) {
    ts_actor_mlp(h, net, m);
    ts_mlp_take(h, N, m, false);
}
// eps[N][A] = actor(x, t, obs); appends to the workspace (the caller may hold pointers below ws.used)
static int ts_actor_forward(dppo_handle* h, cudaStream_t s, int net, const float* x, const float* obs, int obs_div, int N,
                            const int* trow, int tconst, float* eps, int chainK = 0) {
    const Geom& g = h->g; const int KP0 = h->ts->KP0;
    const size_t mark = h->ws.used;
    TsMlp m;
    DPPO_TRY(ws_append(h->ws, [&] { ts_actor_forward_take(h, net, N, m); }));
    m.out = eps;
    // every program of this mode folds, so that the log-prob forward and the update's forward are the same arithmetic and the PPO
    // ratio of unchanged weights is exactly 1 (the full-size parity tests assert it)
    DPPO_TRY(ts_ensure_fold(h, net, s));
    ts_pack_h0_kernel<<<tc_nblk((size_t)N * (KP0 / 8), 256), 256, 0, s>>>(x, obs, trow, tconst, N, g.A, g.Do, g.T, KP0, obs_div, m.h0, split_null(), chainK);
    TC_KCHECK(h);
    const int r = ts_mlp_forward(h, s, m, N);
    h->ws.used = mark;
    return r;
}
static int ts_value(dppo_handle* h, cudaStream_t s, const float* obs, int N, float* v) {
    const Geom& g = h->g; const int KP0 = h->ts->KP0;
    TsMlp m; ts_critic_mlp(h, m);
    DPPO_TRY(ws_layout(h->ws, s, [&] { ts_mlp_take(h, N, m, false); }));
    m.out = v;
    DPPO_TRY(ts_ensure_fold(h, DPPO_NET_CRITIC, s));
    ts_pack_h0_kernel<<<tc_nblk((size_t)N * (KP0 / 8), 256), 256, 0, s>>>(nullptr, obs, nullptr, -1, N, g.A, g.Do, g.T, KP0, 1,
                                                                          m.fp == 4 ? m.h0 : split_null(), m.fp == 4 ? split_null() : m.h0, 0);
    TC_KCHECK(h);
    return ts_mlp_forward(h, s, m, N);
}

// ------------------------------------------------------------------ gradients
// PPODiffusion.c_loss + tape.gradient (diffusion_ppo.py:32-132, train_ppo_diffusion_agent.py:340-346).  Leaves
// [actor_ft grads | critic grads | 8 metrics] in h->grads.  13 plane-GEMM launches + 8 small kernels:
// h0 pack | folded output layers + adv-stats (second stream) | 3 + 3 forward | loss | 3 + 3 backward | grouped dW + reduce | tail || dW3 assembly.
// shapes / alignment the index-driven variant needs (float4 row reads of the resident rollout buffers)
static bool ts_ppo_indexed_ok(const dppo_handle* h, const TcIdxView& v) {
    return loss8_ok(h->g.A, 128, v.chains, v.olp);
}
// idx (optional): the minibatch is given as flat (rollout row, denoising index) indices into the resident rollout buffers; the h0 pack,
// the advantage statistics and the loss kernel address those buffers directly (no gathered copy), the row pointers are unused
static int ts_ppo_step(dppo_handle* h, cudaStream_t s, const float* obs, const float* prev, const float* nxt, const int32_t* inds,
                       const float* returns, const float* oldvalues, const float* advantages, const float* oldlogp,
                       int N, int64_t N_global, float adv_mean, float adv_std, const TcIdxView* idx = nullptr) {
    const Geom& g = h->g; const int KP0 = h->ts->KP0;
    const size_t nA = g.ao.n, nC = g.co.n;
    float* gr = h->grads;
    const bool loss8 = idx ? loss8_ok(g.A, 128, idx->chains, idx->olp) : loss8_ok(g.A, 128, prev, nxt, oldlogp);
    const int NOP = ts_nop(g.A);                                  // the actor's seed width: 64 (A <= 32) or 128
    const bool wide = NOP > 64;                                   // the loss kernel takes a warp per row (tc_ppo_loss8_kernel<32>)
    const int NOg = g.A > 32 ? g.A : 32;                          // columns of the a1^T dout / h0^T dout scratch
    if (idx && !loss8) DPPO_FAIL(-7, "ts_ppo_step: the indexed update needs A %% 4 == 0 and A <= 128");
    const int nlb = loss8 ? tc_nblk(N, wide ? 256 / 32 : LOSS8_ROWS) : tc_nblk(N, 128);
    const int nrb = (N + 31) / 32;
    const size_t pf = ts_part_floats(h, g.H);
    TsMlp ma, mc; ts_actor_mlp(h, DPPO_NET_ACTOR_FT, ma); ts_critic_mlp(h, mc);
    float *eps, *deps, *val, *dval, *part, *dw0a, *dw0c, *colb3, *cpa, *cpc, *gfold; SplitT depsb, dvalb; double* bsum; int* ebeg;
    DPPO_TRY(ws_layout(h->ws, s, [&] {
        ts_mlp_take(h, N, ma, true); ts_mlp_take(h, N, mc, true, false);
        eps = ws_take<float>(h, (size_t)N * g.A); deps = ws_take<float>(h, (size_t)N * g.A);
        val = ws_take<float>(h, N); dval = ws_take<float>(h, N);
        depsb = ts_take(h, (size_t)N * NOP, 2); dvalb = ts_take(h, (size_t)N * 64, 2);
        part = ws_take<float>(h, pf);
        dw0a = ws_take<float>(h, (size_t)KP0 * g.H); dw0c = ws_take<float>(h, (size_t)KP0 * g.Hc);
        bsum = ws_take<double>(h, (size_t)nlb * 5);
        ebeg = ws_take<int>(h, 16);
        colb3 = ws_take<float>(h, (size_t)nlb * (g.A + 1));
        cpa = ws_take<float>(h, (size_t)nrb * 2 * g.H); cpc = ws_take<float>(h, (size_t)nrb * 2 * g.Hc);
        gfold = ws_take<float>(h, (size_t)(g.H + g.Hc + 2 * KP0) * NOg + g.H + g.Hc);      // a1^T dout / h0^T dout of both nets (folded output layer) + scratch
    }));
    float* ga1 = gfold; float* ga0 = ga1 + (size_t)g.H * g.A; float* gc1 = ga0 + (size_t)KP0 * g.A; float* gc0 = gc1 + g.Hc;
    ma.out = eps; mc.out = val;
    // The critic's GEMMs are independent of the actor's until the loss (and again until the weight gradients) and their tiles are
    // short (K = 256: epilogue-latency-bound), while every persistent GEMM leaves SMs idle in its last wave: the critic (and the
    // advantage statistics, which only the loss kernel reads) run on a second stream and fill the actor kernels' tails.
    // (not while the per-kernel profile is on: its event brackets are meant to time each kernel running alone)
    const bool side = !h->prof_on;
    cudaStream_t sc = s;
    if (side) { DPPO_TRY(ensure_aux_stream(h)); sc = h->aux_stream; }
    auto fork = [&]() -> int { if (side) { CUDA_TRY(cudaEventRecord(h->aux_ev[0], s)); CUDA_TRY(cudaStreamWaitEvent(sc, h->aux_ev[0], 0)); } return 0; };
    auto join = [&]() -> int { if (side) { CUDA_TRY(cudaEventRecord(h->aux_ev[1], sc)); CUDA_TRY(cudaStreamWaitEvent(s, h->aux_ev[1], 0)); } return 0; };
    // h0 straight from (prev, obs, K-1-inds): tconst = -(K) flags "t = K-1-trow[r]"; the critic reads the same tile (its x / one-hot rows of W0 are zero)
    // (the actor takes fp16 planes; a smooth critic the bf16 ones written by the same pass, a critic with kinks shares the actor's)
    const SplitT hb = ma.h0b;                                   // bf16 copy: the weight-gradient operand, and a smooth critic's input
    if (mc.fp != 4) mc.h0 = ma.h0b;
    if (idx) ts_pack_h0_kernel<<<tc_nblk((size_t)N * (KP0 / 8), 256), 256, 0, s>>>(idx->chains, idx->obs, nullptr, 0, N, g.A, g.Do, g.T, KP0, 1, ma.h0, hb, 0,
                                                                                     idx->flat, idx->K, idx->P, idx->bad);
    else ts_pack_h0_kernel<<<tc_nblk((size_t)N * (KP0 / 8), 256), 256, 0, s>>>(prev, obs, inds, -g.K, N, g.A, g.Do, g.T, KP0, 1, ma.h0, hb, 0);
    TC_KCHECK(h);
    if (mc.fp == 4) { mc.h0 = ma.h0; mc.h0b = ma.h0b; }
    // The actor's two big layers are handed to the GPU before the host enqueues the second stream's kernels: after a step that ended with
    // the metrics on the host the device is idle, and the short first kernels would otherwise run at the host's launch rate.
    if (side) {
        CUDA_TRY(cudaEventRecord(h->aux_ev[0], s));
        DPPO_TRY(ts_mlp_forward(h, s, ma, N, 1));
        CUDA_TRY(cudaStreamWaitEvent(sc, h->aux_ev[0], 0));
    }
    // the folded output layers of the current weights (stale after every AdamW step): on the second stream, under the actor's L0 / L1
    DPPO_TRY(ts_ensure_fold(h, DPPO_NET_ACTOR_FT, sc)); DPPO_TRY(ts_ensure_fold(h, DPPO_NET_CRITIC, sc));
    if (side) { CUDA_TRY(cudaEventRecord(h->aux_ev[2], sc)); ma.fold_ev = h->aux_ev[2]; }      // the actor's stream waits in front of its folded GEMM only
    DPPO_TRY(launch_adv_stats(h, sc, advantages, idx, N, adv_mean, adv_std));
    DPPO_TRY(ts_mlp_forward(h, s, ma, N, side ? 2 : 0));
    DPPO_TRY(ts_mlp_forward(h, sc, mc, N));
    DPPO_TRY(join());
    const PpoHyper hp = ppo_hyper(h, N_global);
    const float frac_local = (float)((double)N / (double)N_global);
    if (loss8) {
        // loss, metric partial sums, the two-plane padded gradient seeds and the output-bias column partials in one pass
        TcIdxView iv; memset(&iv, 0, sizeof(iv));
        if (idx) iv = *idx;
        auto loss = wide ? tc_ppo_loss8_kernel<32> : tc_ppo_loss8_kernel<8>;
        loss<<<nlb, 256, 0, s>>>(prev, nxt, eps, inds, returns, oldvalues, advantages, oldlogp, val, h->scalars, h->sched, hp, N,
                                 depsb.p[0], dvalb.p[0], bsum, colb3, iv, depsb.p[1], dvalb.p[1]);
        TC_KCHECK(h);
    } else {
        ppo_loss_kernel<<<nlb, 128, 0, s>>>(prev, nxt, eps, inds, returns, oldvalues, advantages, oldlogp, val, h->scalars, h->sched, hp, N, deps, dval, bsum);
        TC_KCHECK(h);
        ts_pad64_kernel<<<tc_nblk((size_t)N * (NOP / 8), 256), 256, 0, s>>>(deps, N, g.A, NOP, depsb.p[0], depsb.p[1]); TC_KCHECK(h);
        ts_pad64_kernel<<<tc_nblk((size_t)N * 8, 256), 256, 0, s>>>(dval, N, 1, 64, dvalb.p[0], dvalb.p[1]); TC_KCHECK(h);
    }
    // both backward chains, then ONE grouped launch with the eight weight-gradient products of actor and critic
    DPPO_TRY(fork());
    DPPO_TRY(ts_mlp_backward_dx(h, s, ma, depsb, N, cpa));
    DPPO_TRY(ts_mlp_backward_dx(h, sc, mc, dvalb, N, cpc));
    DPPO_TRY(join());
    tsp::DwDesc dd[10];
    const int nda = ts_mlp_dw_descs(ma, depsb, N, gr, g.ao.w1, dw0a, dd, ga1, ga0);
    const int ndc = ts_mlp_dw_descs(mc, dvalb, N, gr + nA, g.co.w1, dw0c, dd + nda, gc1, gc0);
    DPPO_TRY(tsp::launch_dw_pair(h, s, dd, nda + ndc, N, part, pf, ebeg));
    // everything dv would have fed (dW3, dW2, db2, the residual share of dw0) from the two small products; before the tail, which reads dw0
    // (the dw0 / db2 rows first, on this stream; dW3 and dW2 - which only AdamW reads - beside the tail kernel on the second stream)
    DPPO_TRY(ts_dw3_assemble(h, s, DPPO_NET_ACTOR_FT, ga1, ga0, gr, dw0a, gc1, gc0, gr + nA, dw0c, 0));
    DPPO_TRY(fork());
    DPPO_TRY(ts_dw3_assemble(h, sc, DPPO_NET_ACTOR_FT, ga1, ga0, gr, dw0a, gc1, gc0, gr + nA, dw0c, 1));
    float* b2scr = gfold + (size_t)(g.H + g.Hc + 2 * KP0) * NOg;     // the unwritten slot-0 column sums land here, not in db2
    if (loss8) {
        DPPO_TRY(tc_launch_tail(h, s, bsum, nlb, hp.inv_nglobal, frac_local, colb3, cpa, nrb, cpc, nrb, dw0a, dw0c, b2scr, b2scr + g.H));
        DPPO_TRY(join());
        return 0;
    }
    DPPO_TRY(join());
    // (unaligned / wide action rows) the same pieces as separate launches
    ppo_metrics_kernel<<<1, 256, 0, s>>>(bsum, nlb, hp.inv_nglobal, frac_local, gr + nA + nC); TC_KCHECK(h);
    DPPO_TRY(colsum(h, s, deps, g.A, N, g.A, nullptr, 1, part, gr + g.ao.b3));
    DPPO_TRY(colsum(h, s, dval, 1, N, 1, nullptr, 1, part, gr + nA + g.co.b3));
    tc_reduce_cols_kernel<<<tc_nblk(2 * g.H, 8), 256, 0, s>>>(cpa, nrb, (size_t)2 * g.H, 2 * g.H, b2scr, g.H, gr + g.ao.b1); TC_KCHECK(h);
    tc_reduce_cols_kernel<<<tc_nblk(2 * g.Hc, 8), 256, 0, s>>>(cpc, nrb, (size_t)2 * g.Hc, 2 * g.Hc, b2scr + g.H, g.Hc, gr + nA + g.co.b1); TC_KCHECK(h);
    return tc_scatter_dw0(h, s, DPPO_NET_ACTOR_FT, dw0a, dw0c, gr);
}

// DiffusionModel.c_loss / p_losses (diffusion.py:179-202) + tape.gradient: loss -> h->grads[nA], gradients -> h->grads[0 : nA]
static int ts_pretrain_grads(dppo_handle* h, cudaStream_t s, const float* actions, const float* obs, int N, int64_t N_global,
                             int64_t row_offset, const int32_t* t_in, const float* noise_in, uint64_t seed, uint64_t offset) {
    const Geom& g = h->g; const int KP0 = h->ts->KP0;
    const size_t nA = g.ao.n; float* gr = h->grads;
    const size_t ne = (size_t)N * g.A;
    const int nlb = tc_nblk(ne, 256);
    const int nrb = (N + 31) / 32;
    const int NOP = ts_nop(g.A), NOg = g.A > 32 ? g.A : 32;
    const size_t pf = ts_part_floats(h, g.H);
    TsMlp ma; ts_actor_mlp(h, DPPO_NET_ACTOR, ma);
    float *ga1, *eps, *deps, *noise, *xn, *part, *dw0, *cpa; int *trow, *ebeg; SplitT depsb; double* bsum;
    DPPO_TRY(ws_layout(h->ws, s, [&] {
        ts_mlp_take(h, N, ma, true);
        ga1 = ws_take<float>(h, (size_t)(g.H + KP0) * NOg + g.H);    // + scratch for the unwritten slot-0 sums
        eps = ws_take<float>(h, ne); deps = ws_take<float>(h, ne); noise = ws_take<float>(h, ne); xn = ws_take<float>(h, ne);
        trow = ws_take<int>(h, N);
        depsb = ts_take(h, (size_t)N * NOP, 2);
        part = ws_take<float>(h, pf);
        dw0 = ws_take<float>(h, (size_t)KP0 * g.H);
        bsum = ws_take<double>(h, nlb);
        ebeg = ws_take<int>(h, 16);
        cpa = ws_take<float>(h, (size_t)nrb * 2 * g.H);
    }));
    float* ga0 = ga1 + (size_t)g.H * g.A;
    DPPO_TRY(ts_ensure_fold(h, DPPO_NET_ACTOR, s));
    ma.out = eps;
    pretrain_prep_kernel<<<tc_nblk(ne, 256), 256, 0, s>>>(actions, t_in, noise_in, N, g.A, g.T, h->sched, seed, offset, row_offset, trow, noise, xn); TC_KCHECK(h);
    ts_pack_h0_kernel<<<tc_nblk((size_t)N * (KP0 / 8), 256), 256, 0, s>>>(xn, obs, trow, 0, N, g.A, g.Do, g.T, KP0, 1, ma.h0, ma.h0b, 0); TC_KCHECK(h);
    DPPO_TRY(ts_mlp_forward(h, s, ma, N));
    const float scale = 1.0f / ((float)N_global * (float)g.A);
    mse_loss_kernel<<<nlb, 256, 0, s>>>(eps, noise, ne, scale, deps, bsum); TC_KCHECK(h);
    sum_blocks_kernel<<<1, 256, 0, s>>>(bsum, nlb, scale, gr + nA); TC_KCHECK(h);
    ts_pad64_kernel<<<tc_nblk((size_t)N * (NOP / 8), 256), 256, 0, s>>>(deps, N, g.A, NOP, depsb.p[0], depsb.p[1]); TC_KCHECK(h);
    DPPO_TRY(ts_mlp_backward_dx(h, s, ma, depsb, N, cpa));
    tsp::DwDesc dd[5];
    const int nd = ts_mlp_dw_descs(ma, depsb, N, gr, g.ao.w1, dw0, dd, ga1, ga0);
    DPPO_TRY(tsp::launch_dw_pair(h, s, dd, nd, N, part, pf, ebeg));
    DPPO_TRY(ts_dw3_assemble(h, s, DPPO_NET_ACTOR, ga1, ga0, gr, dw0, nullptr, nullptr, nullptr, nullptr));
    tc_reduce_cols_kernel<<<tc_nblk(2 * g.H, 8), 256, 0, s>>>(cpa, nrb, (size_t)2 * g.H, 2 * g.H, ga1 + (size_t)(g.H + KP0) * NOg, g.H, gr + g.ao.b1); TC_KCHECK(h);
    DPPO_TRY(colsum(h, s, deps, g.A, N, g.A, nullptr, 1, part, gr + g.ao.b3));
    return tc_scatter_dw0(h, s, DPPO_NET_ACTOR, dw0, nullptr, gr);
}
