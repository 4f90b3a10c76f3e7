// Grouped weight-gradient GEMM on CTA pairs (cta_group::2):  out_p[M_p][N_p] += X_p^T D_p  for up to 10 problems, ONE launch.
//
// All problems reduce over the same rows (K = rows of the chunk); X_p [rows][M_p] and D_p [rows][N_p] are bf16 row-major
// (both operands MN-major).  Every CTA pair takes (output tile, K split) work items from a flat list; the number of splits
// per problem is chosen on the host so that the items have equal cost and fill the SMs once.  Partial tiles are accumulated
// with red.global.add (outputs zeroed by the caller).
// A CTA pair owns a 256 x 256 (or 256 x 128) output tile.  Each CTA stages its own 128 columns of X and only HALF of the
// D tile per 64-row k-block (32 KB instead of the 48 KB of a lone 128 x 256 CTA), the leader issues 256-row tcgen05.mma
// that read the two D halves from both CTAs' shared memory.  A single CTA sits at the ~34 B/cycle/SM TMA ingest limit
// (DESIGN.md 5.2: 96 B/cycle wanted); the pair needs 64 B/cycle for the same MMA rate.
//
// Narrow problems are given with the wide operand as X: the layer-0 products h0^T du / h0^T dv arrive as du^T h0
// (M = H, N = 64) and are written transposed.  N = 64 problems run as N = 128 (the second CTA's half is out of bounds and
// zero-filled by TMA), so that the per-CTA D box keeps the 128-byte swizzle.
#pragma once
#include "fused_chain.cuh"

namespace tcp {
using namespace tc;
constexpr int GMAX = 10, PSTAGES = 6, PBK = 64;
struct GroupMaps { CUtensorMap a[GMAX]; CUtensorMap b[GMAX]; };
constexpr int PA_STAGE = 128 * PBK * 2, PB_STAGE = 128 * PBK * 2;     // per CTA: 128 X columns, <= 128 D columns
struct PairProb {
    int m_blocks, n_blocks;           // 256-row output blocks; 256-column (or 128-column) blocks
    int nb_cta;                       // 64-column D boxes per CTA per k-block (2: N tile 256, 1: N tile 128)
    int splits, kb_per_split, item_begin;
    int M_valid, N_valid, ld_out, transposed;
    float* out;
};
struct PairParams { int nprob, items, kblocks; PairProb p[GMAX]; };
constexpr size_t pair_smem_bytes() { return (size_t)PSTAGES * (PA_STAGE + PB_STAGE) + 1024 + 256; }

__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}"
                 ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}

__global__ void __launch_bounds__(NUM_THREADS, 1) dw_pair_kernel(const __grid_constant__ GroupMaps maps, const PairParams gp) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* sA = smem;
    uint8_t* sB = smem + PSTAGES * PA_STAGE;
    uint64_t* bars = (uint64_t*)(smem + PSTAGES * (PA_STAGE + PB_STAGE));
    uint64_t* full = bars;                      // leader's: both CTAs' producers + their TMA bytes
    uint64_t* empty = bars + PSTAGES;           // per CTA: multicast commit of the MMAs that read the stage
    uint64_t* tfull = bars + 2 * PSTAGES;       // per CTA: multicast commit, accumulator complete
    uint64_t* tempty = tfull + 2;               // leader's: the 8 epilogue warps of the pair drained the accumulator
    uint32_t* tmem_slot = (uint32_t*)(tempty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = fc::cluster_ctarank();
    const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < PSTAGES; ++i) { mbar_init(&full[i], 2); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 8); }
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

    auto decode = [&](int item, int& pi, int& m_blk, int& n_blk, int& split) {
        pi = 0;
        while (pi + 1 < gp.nprob && item >= gp.p[pi + 1].item_begin) ++pi;
        const PairProb& P = gp.p[pi];
        const int local = item - P.item_begin, per = P.m_blocks * P.n_blocks;
        split = local / per; const int rem = local % per;
        m_blk = rem / P.n_blocks; n_blk = rem % P.n_blocks;
    };

    if (warp == 0) {
        // ---- TMA producer (both CTAs): own X columns, own half of the D tile; bytes and arrival go to the leader's barrier
        int stage = 0; uint32_t phase = 0;
        const uint32_t a_addr = smem_u32(sA), b_addr = smem_u32(sB), full_addr = smem_u32(full);
        for (int item = pair; item < gp.items; item += npairs) {
            int pi, m_blk, n_blk, split; decode(item, pi, m_blk, n_blk, split);
            const PairProb& P = gp.p[pi];
            const int kb0 = split * P.kb_per_split, kb1 = min(gp.kblocks, kb0 + P.kb_per_split);
            const uint32_t tx = (uint32_t)(PA_STAGE + P.nb_cta * 64 * PBK * 2);
            const int m0 = m_blk * 256 + (int)rank * 128, n0 = n_blk * (P.nb_cta * 128) + (int)rank * (P.nb_cta * 64);
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(&empty[stage], phase ^ 1);
                if (elect_one_lane()) {
                    const uint32_t fb = full_addr + stage * 8;
                    fc::mbar_expect_tx_cluster(fc::mapa_rank0(fb), tx);
                    const uint32_t a = a_addr + stage * PA_STAGE, b = b_addr + stage * PB_STAGE;
                    fc::tma_load_2d_pair(a, &maps.a[pi], fb, m0, kb * PBK);
                    fc::tma_load_2d_pair(a + 64 * PBK * 2, &maps.a[pi], fb, m0 + 64, kb * PBK);
                    for (int j = 0; j < P.nb_cta; ++j) fc::tma_load_2d_pair(b + j * (64 * PBK * 2), &maps.b[pi], fb, n0 + j * 64, kb * PBK);
                }
                __syncwarp();
                if (++stage == PSTAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ---- MMA issuer: the leader only
        if (rank == 0) {
            int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
            for (int item = pair; item < gp.items; item += npairs) {
                int pi, m_blk, n_blk, split; decode(item, pi, m_blk, n_blk, split);
                const PairProb& P = gp.p[pi];
                const int kb0 = split * P.kb_per_split, kb1 = min(gp.kblocks, kb0 + P.kb_per_split);
                const uint32_t idesc = make_idesc(256, P.nb_cta * 128, true, true);
                mbar_wait(&tempty[acc], acc_phase ^ 1);
                tcgen05_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * 256);
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tcgen05_fence_after();
                    const uint32_t a0 = smem_u32(sA + stage * PA_STAGE), b0 = smem_u32(sB + stage * PB_STAGE);
                    if (elect_one_lane()) {
#pragma unroll
                        for (int k = 0; k < PBK / 16; ++k)
                            umma_bf16_pair(tmem_d, make_desc(a0 + k * 2048, 64 * PBK * 2, 1024), make_desc(b0 + k * 2048, 64 * PBK * 2, 1024), idesc,
                                           (kb > kb0 || k > 0) ? 1u : 0u);
                        fc::tcgen05_commit_pair(smem_u32(&empty[stage]));
                    }
                    __syncwarp();
                    if (++stage == PSTAGES) { stage = 0; phase ^= 1; }
                }
                if (elect_one_lane()) fc::tcgen05_commit_pair(smem_u32(&tfull[acc]));
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ---- epilogue (both CTAs): own 128 rows x the full N tile, accumulated into the gradient with vector reds
        const int quad = warp & 3;
        int acc = 0; uint32_t acc_phase = 0;
        const uint32_t tempty_leader = fc::mapa_rank0(smem_u32(tempty));
        for (int item = pair; item < gp.items; item += npairs) {
            int pi, m_blk, n_blk, split; decode(item, pi, m_blk, n_blk, split);
            const PairProb& P = gp.p[pi];
            mbar_wait(&tfull[acc], acc_phase);
            tcgen05_fence_after();
            const int m = m_blk * 256 + (int)rank * 128 + quad * 32 + lane;
            const bool row_ok = m < P.M_valid;
            const int ntile = P.nb_cta * 128;
#pragma unroll 1
            for (int c = 0; c < ntile / 32; ++c) {
                const int n0 = n_blk * ntile + c * 32;
                if (n0 >= P.N_valid) break;                                  // warp-uniform
                uint32_t r[32];
                tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * 256 + c * 32), r);
                if (!row_ok) continue;
                if (P.transposed) {
                    // out[n][m]: the 32 lanes of a warp hold consecutive m -> one coalesced red per column
                    for (int j = 0; j < 32; ++j) if (n0 + j < P.N_valid) atomicAdd(P.out + (size_t)(n0 + j) * P.ld_out + m, __uint_as_float(r[j]));
                } else {
                    float* dst = P.out + (size_t)m * P.ld_out + n0;
                    if (n0 + 32 <= P.N_valid && (P.ld_out & 3) == 0 && ((uintptr_t)dst & 15) == 0) {   // (a net's slice of the flat gradient need not start 16-byte aligned)
#pragma unroll
                        for (int q = 0; q < 8; ++q)
                            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + q * 4), "f"(__uint_as_float(r[q * 4])), "f"(__uint_as_float(r[q * 4 + 1])),
                                         "f"(__uint_as_float(r[q * 4 + 2])), "f"(__uint_as_float(r[q * 4 + 3])) : "memory");
                    } else {
                        for (int j = 0; j < 32; ++j) if (n0 + j < P.N_valid) atomicAdd(dst + j, __uint_as_float(r[j]));
                    }
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) fc::mbar_arrive_cluster(tempty_leader + acc * 8);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    fc::cluster_sync_all();                     // the peer may still be signalling our barriers / reading our D halves
    if (warp == 1) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// one problem: out += X^T D with X [rows][M], D [rows][Nd]; transposed: out[n][m] (ld_out = row length of that layout)
struct PairDesc { const __nv_bfloat16* X; int M; const __nv_bfloat16* D; int Nd; float* out; int M_valid, N_valid, ld_out, transposed; double alg_flops; };

static int launch_group_pair(dppo_handle* h, cudaStream_t s, const PairDesc* d, int n, int rows) {
    if (h->sm_count < 2 || n < 1 || n > GMAX) DPPO_FAIL(-1, "launch_group_pair: bad problem count %d", n);
    for (int i = 0; i < n; ++i) if (d[i].M % 64 || d[i].Nd % 64) DPPO_FAIL(-7, "launch_group_pair: operand widths must be multiples of 64");
    GroupMaps maps; PairParams gp; memset(&gp, 0, sizeof(gp));
    gp.nprob = n; gp.kblocks = (rows + PBK - 1) / PBK;
    const int npairs = h->sm_count / 2;
    double w[GMAX]; int tiles[GMAX];
    const double w128 = 0.75;                  // relative k-block time of a 128-wide tile (24 KB staged per CTA vs 32 KB)
    for (int i = 0; i < n; ++i) {
        PairProb& P = gp.p[i];
        DPPO_TRY(make_map(&maps.a[i], d[i].X, rows, d[i].M, d[i].M, PBK, 64));
        DPPO_TRY(make_map(&maps.b[i], d[i].D, rows, d[i].Nd, d[i].Nd, PBK, 64));
        P.m_blocks = (d[i].M + 255) / 256;
        const int nb64 = (d[i].Nd + 63) / 64;
        P.nb_cta = nb64 <= 2 ? 1 : 2;
        P.n_blocks = (nb64 + 2 * P.nb_cta - 1) / (2 * P.nb_cta);              // tile width = nb_cta * 128 columns
        P.M_valid = d[i].M_valid; P.N_valid = d[i].N_valid; P.ld_out = d[i].ld_out; P.out = d[i].out; P.transposed = d[i].transposed;
        tiles[i] = P.m_blocks * P.n_blocks;
        w[i] = P.nb_cta == 2 ? 1.0 : w128;
    }
    for (int i = n; i < GMAX; ++i) { maps.a[i] = maps.a[0]; maps.b[i] = maps.b[0]; }
    // K splits: the smallest per-item budget (in 256-wide k-block units) for which all items fit the pairs in ONE wave
    auto items_for = [&](double budget) { int it = 0; for (int i = 0; i < n; ++i) { int sp = (int)ceil(gp.kblocks * w[i] / budget); if (sp < 1) sp = 1; it += tiles[i] * sp; } return it; };
    double lo = 4.0, hi = (double)gp.kblocks;
    if (items_for(lo) <= npairs) hi = lo;
    for (int it = 0; it < 40 && hi - lo > 0.25; ++it) { const double mid = 0.5 * (lo + hi); if (items_for(mid) <= npairs) hi = mid; else lo = mid; }
    int items = 0; double flops = 0;
    for (int i = 0; i < n; ++i) {
        PairProb& P = gp.p[i];
        int splits = (int)ceil(gp.kblocks * w[i] / hi);
        if (splits < 1) splits = 1;
        if (splits > gp.kblocks) splits = gp.kblocks;
        P.kb_per_split = (gp.kblocks + splits - 1) / splits;
        P.splits = (gp.kblocks + P.kb_per_split - 1) / P.kb_per_split;
        P.item_begin = items; items += tiles[i] * P.splits;
        flops += d[i].alg_flops;
    }
    gp.items = items;
    static bool attr_set_dev[64] = {};      // function attributes are per device
    bool& attr_set = attr_set_dev[h->device & 63];
    if (!attr_set) {
        CUDA_TRY(cudaFuncSetAttribute(dw_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pair_smem_bytes()));
        attr_set = true;
    }
    const int grid = 2 * (items < npairs ? items : npairs);
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1; cfg.blockDim = dim3(NUM_THREADS); cfg.gridDim = dim3(grid); cfg.dynamicSmemBytes = pair_smem_bytes(); cfg.stream = s;
    prof_begin(h, s);
    cudaError_t le = cudaLaunchKernelEx(&cfg, dw_pair_kernel, maps, gp);
    prof_end(h, s, flops, 1);
    h->launches++; h->tc_launches++;
    if (le != cudaSuccess) DPPO_FAIL(-3, "grouped dW (pair) launch failed: %s", cudaGetErrorString(le));
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) DPPO_FAIL(-3, "grouped dW (pair) launch failed: %s", cudaGetErrorString(e));
    return 0;
}
}  // namespace tcp
