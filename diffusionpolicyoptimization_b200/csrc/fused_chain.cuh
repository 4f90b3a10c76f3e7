// Fused residual-MLP layer chain on tcgen05 (sm_100a).  A persistent CTA PAIR (cluster of 2, cta_group::2) walks
// 256-row tiles - 128 rows per CTA - and runs EVERY layer of the chain for its tile with the activations resident on chip.
//
//   shared memory  X   [128][H] bf16   the current activation, stored as H/64 K-major 128B-swizzled tiles
//   (per CTA)                          (exactly the image TMA would produce), i.e. directly the A operand
//                                      of the next layer's tcgen05.mma and the source of a TMA store
//                  G   [128][H] bf16   (H = 256 only) Mish gates mish'(pre-activation): written next to X in the
//                                      forward pass (TMA-stored for the backward), TMA-loaded in the backward pass
//                  H0  [128][64] bf16  the packed layer-0 input tile [x | obs | onehot(t) | 1 | 0]
//                                      (TMA-loaded, or rebuilt in place by the sampler every denoising step)
//                  W   4 x 16 KB ring  this CTA's half of every weight tile: [64 k][128 n] (MN-major, TMA from L2);
//                                      the pair's MMA reads both halves
//   tensor memory  512 columns         the whole [128][H] fp32 accumulator of one layer
//
//   warp 0     TMA producer (weight ring, H0 / gate tiles); loads report to the LEADER CTA's mbarriers
//   warp 1     tcgen05.mma issuer (leader CTA only, warp-uniform + elect.sync), TMEM allocation
//   warps 2-9  epilogue (two warps per TMEM lane quadrant; software-pipelined tcgen05.ld): bias / ReLU (+ bit mask) /
//              Mish (+ gate) / mask or gate multiply -> bf16 -> swizzled st.shared into X (+ TMA store of X to HBM
//              when the backward pass needs the tensor, + bias-gradient column sums), and the final-layer math:
//              eps / value store, Gaussian log-prob, or the DDPM posterior step of the sampler.
//
// A 512-wide layer is drained in two phases so that epilogue and MMA overlap: columns [0,256) while the second n-half's
// MMAs still run (X tile j is overwritten only once those MMAs consumed it: xfree[j]); the next layer's MMAs start on
// X tiles [0, XT/2) while phase two still writes the rest (xready[0/1], acc_full[0/1]).  Programs on this engine:
//   forward   L0 act(H0 W0 + b0) -> L1 act(X W1 + b1) -> L2 X W2 + H0 W0 + b2 (residual by K-concatenation)
//             -> L3 X W3 + b3 ;  final = output store | log-prob | (training) + stored a0, a1, v + masks / gates
//   backward  B1 dv = dout W3^T -> B2 dh1 = (dv W2^T) . act'(h1) -> B3 du = (dh1 W1^T) . act'(u)   (each stored by TMA)
//   sampler   T denoising steps x forward, x kept in the epilogue threads' registers, noise from Philox
//             (or injected), chain / actions written once: ONE launch per rollout step.
#pragma once
#include "tc_gemm.cuh"
#include "simt_kernels.cuh"

namespace fc {
using namespace tc;

constexpr int FBM = 128, WK = 32, NSTAGE = 4, FTHREADS = 320, MAXL = 4, NMAPS = 10;   // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue
constexpr int STAGE_BYTES = WK * 256 * 2;      // 16 KB
constexpr int H0_BYTES = FBM * 64 * 2;         // 16 KB

enum { FINAL_STORE = 0, FINAL_EPS = 1, FINAL_LOGP = 2, FINAL_SAMPLE = 3 };

struct Layer {
    int a_src;                 // 0: H0 tile only (K = 64); 1: X (K = H); 2: X then H0 (K = H + 64)
    int wmap;                  // tensor map of the B operand: bf16 [K][N] (MN-major), box [WK][64]
    int wrow_x, wrow_h0;       // first k-row of the X part / the H0 part inside that map
    int n;                     // output width: H, or 64 for the output layer
    int h0_last;               // this layer is the tile's last reader of H0 (TMA mode): release it afterwards
    const float* bias;         // [n] fp32 or null
    int act;                   // 0 none, 1 ReLU, 2 Mish
    const uint32_t* mask_in;   // [rows][H/32] ReLU bit masks to multiply with, or null
    uint32_t* mask_out;        // [rows][H/32] ReLU bit masks to record, or null
    int store_map;             // tensor map for the TMA store of X ([rows][H] bf16, box [128][64]), or -1
    // Mish networks (H = 256 only: a second [128][H] buffer G lives next to X)
    int gate_store_map;        // act == 2: also store G = mish'(pre-activation) ([rows][H] bf16) for the backward pass, or -1
    int gate_load_map;         // backward: multiply by the gate tile TMA-loaded from this map into G, or -1
    int colsum_slot;           // 0 / 1: accumulate the column sums of this layer's stored X (bias gradient), or -1
};

struct Params {
    int rows, nlayers, final_mode, h0_from_tma;
    Layer L[2][MAXL];          // [net][layer]; net 1 = fine-tuned actor (sampler only)
    int A, Do, T, K;
    const float* sch;
    // FINAL_EPS / FINAL_LOGP
    float* out;                // eps [rows][A] or logp [rows][A]
    const float* prev; const float* next; const float* chains; const int* trow;
    float dcv, min_lp_std;
    // FINAL_SAMPLE
    const float* obs; const float* xT; const float* noise;
    float* actions; float* chains_out;
    SampleHyper hp; int use_base_policy;
    uint64_t seed, offset; int64_t row_offset;
    float* colsum_part;        // [grid][2][H] per-CTA column sums of the layers with colsum_slot >= 0 (bias gradients)
    long long* dbg;            // optional [grid][8] cycle counters (dev tool): see chain_kernel
};
struct Maps { CUtensorMap m[NMAPS]; };

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void epi_barrier() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void ld_shared_v4(uint32_t addr, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr) : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&t);
}

// Mish and its derivative from one exponential: with n = e^x, w = n^2 + 2n:  tanh(softplus(x)) = w / (w + 2),
// d/dx = 4 n (n + 1) / (w + 2)^2.  (tensor path only; the fp32 parity path keeps the literal x * tanh(softplus(x)))
__device__ __forceinline__ void mish_and_grad(float x, float& y, float& g) {
    // flush-to-zero approximations without the denormal range fix-ups nvcc adds around __expf / __fdividef; the
    // clamp at 20 keeps w finite and the formulas already give y = x, g = 1 to fp32 precision there
    float n, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(n) : "f"(fminf(x, 20.f) * 1.4426950408889634f));
    const float w = fmaf(n, n, n + n);
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(w + 2.f));
    const float f = w * r;
    y = x * f;
    g = fmaf(4.f * x, fmaf(n, n, n) * r * r, f);
}
// One lane of a converged warp (elect.sync).  The issue warps keep warp-uniform control flow and elect a lane only
// around the tcgen05 / TMA instructions: inside a lane-divergent branch (`if (lane == 0)`) nvcc wraps every
// uniform-datapath instruction (UTCHMMA, UTCBAR, UTMALDG) in an ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall loop,
// which made the single issuing thread the bottleneck (tools/mma_probe.py: ~90 cycles per tcgen05.mma issued).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P1;\n\telect.sync _|P1, 0xFFFFFFFF;\n\tselp.b32 %0, 1, 0, P1;\n\t}" : "=r"(pred));
    return pred != 0;
}
// raw shared-address variants for the single-thread issue loops (no generic->shared conversion per call)
__device__ __forceinline__ bool mbar_try_wait_addr(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_addr(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait_addr(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait_addr(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) { printf("fused chain: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x); __trap(); }
    }
}
__device__ __forceinline__ void mbar_expect_tx_addr(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d_addr(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tcgen05_commit_addr(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// tcgen05.mma with the two shared-memory descriptors given as (low word, shared high word)
__device__ __forceinline__ void umma_bf16_split(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tmov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\tsetp.ne.b32 p, %5, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}"
                 ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(accumulate) : "memory");
}

// ---- CTA-pair (cta_group::2) helpers: the two CTAs of a cluster form one 256-row MMA; each holds its own 128 rows of A
// and half of every B tile, the leader (rank 0) issues the MMAs and both CTAs' TMA loads report to the leader's barriers
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_rank0(uint32_t addr) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(0)); return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_cluster(uint32_t cluster_addr, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_addr), "r"(bytes) : "memory");
}
// TMA load whose completion bytes are reported to the mbarrier at the same offset in the pair's leader CTA
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_bf16_split_pair(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tmov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\tsetp.ne.b32 p, %5, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, {%6, %6, %6, %6, %6, %6, %6, %6}, p;\n\t}"
                 ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
// commit that arrives on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void tcgen05_commit_pair(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3) : "memory");
}

template <int H> constexpr size_t chain_smem_bytes() {
    return (size_t)(H / 64) * 16384 * (H == 256 ? 2 : 1) + H0_BYTES + (size_t)NSTAGE * STAGE_BYTES + 2 * 512 * sizeof(float) + 1024 + 256;
}

// asynchronous TMEM load of 32 columns (no wait) and the matching wait, tied to the destination registers so
// that no use of them can be scheduled ahead of the wait
__device__ __forceinline__ void tmem_ld32_async(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
          "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
          "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
          "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
        :: "memory");
}
__device__ __forceinline__ void tmem_ld8_async(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait8(uint32_t (&r)[8]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]) :: "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
          "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
        :: "memory");
}

// H0 row image [x (A) | obs (Do) | onehot(t) (T) | 1 | 0..] (64 bf16, 128B-swizzled).  The two epilogue threads of a
// row split it: half 0 owns x[0:16) and writes 16-byte chunks {0,1,4,5}; half 1 owns x[16:32) and writes {2,3,6,7}.
__device__ __forceinline__ void build_h0_half(uint32_t h0_addr, int rloc, int half, const float (&x)[16], const float* __restrict__ obs_row,
                                              int A, int Do, int T, int t, bool valid) {
#pragma unroll
    for (int ci = 0; ci < 4; ++ci) {
        const int c = (ci < 2 ? 0 : 4) + half * 2 + (ci & 1);         // chunk index 0..7
        uint32_t w[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float v2[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int k = c * 8 + j * 2 + e;                      // column
                const int xi = (ci & 1) * 8 + j * 2 + e;              // index into this half's x (only meaningful for ci < 2)
                float v = 0.f;
                if (valid) {
                    if (ci < 2 && k < A) v = x[xi];
                    else if (k >= A && k < A + Do) v = __ldg(obs_row + (k - A));
                    else if (k >= A + Do && k < A + Do + T) v = (k - A - Do == t) ? 1.f : 0.f;
                    else if (k == A + Do + T) v = 1.f;
                }
                v2[e] = v;
            }
            w[j] = pack_bf16(v2[0], v2[1]);
        }
        st_shared_v4(h0_addr + rloc * 128 + ((c ^ (rloc & 7)) << 4), w[0], w[1], w[2], w[3]);
    }
}

template <int H, bool TIMING>
__global__ void __launch_bounds__(FTHREADS, 1) chain_kernel(const __grid_constant__ Maps maps, const Params p) {
    constexpr int XT = H / 64;
    constexpr int WKE = WK * 2;                                 // k-rows per ring stage: a stage is [WKE][128] = 16 KB per CTA
    constexpr int MPS = WKE / 16;                               // tcgen05.mma (K = 16) per stage
    constexpr int X_BYTES = XT * 16384;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* sX = smem;
    constexpr bool HASG = (H == 256);                           // room for the gate buffer next to X
    uint8_t* sG = sX + X_BYTES;
    uint8_t* sH0 = sG + (HASG ? X_BYTES : 0);
    uint8_t* sW = sH0 + H0_BYTES;
    float* sBias = (float*)(sW + NSTAGE * STAGE_BYTES);           // 2 x 512 fp32, double buffered across layers
    uint64_t* bars = (uint64_t*)(sBias + 2 * 512);
    uint64_t* w_full = bars;
    uint64_t* w_empty = bars + NSTAGE;
    uint64_t* h0_full = bars + 2 * NSTAGE;
    uint64_t* h0_empty = h0_full + 1;
    uint64_t* acc_full = h0_full + 2;    // [2] MMA -> epilogue: accumulator columns [256 h, 256 h + 256) complete
    uint64_t* xready = h0_full + 4;      // [2] epilogue -> MMA: X tiles of half h written + TMEM columns of half h drained
    uint64_t* xfree = h0_full + 6;       // [4] MMA -> epilogue: the last n-half has consumed X tile j (j < XT/2)
    uint64_t* g_full = h0_full + 10;     // TMA -> epilogue: gate tile landed in G
    uint64_t* g_empty = h0_full + 11;    // epilogue -> TMA: G may be overwritten
    uint32_t* tmem_slot = (uint32_t*)(h0_full + 12);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ntiles = (p.rows + FBM - 1) / FBM;
    const uint32_t rank = cluster_ctarank();                     // rank inside the CTA pair (leader = 0)
    const int pair0 = blockIdx.x / 2, npairs = gridDim.x / 2, ptiles = (ntiles + 1) / 2;
    const bool sampler = p.final_mode == FINAL_SAMPLE;
    const int nsteps = sampler ? p.T : 1;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < NMAPS; ++i) tma_prefetch_desc(&maps.m[i]);
        for (int i = 0; i < NSTAGE; ++i) { mbar_init(&w_full[i], 2); mbar_init(&w_empty[i], 1); }
        mbar_init(h0_full, 2); mbar_init(h0_empty, 1);
        mbar_init(&acc_full[0], 1); mbar_init(&acc_full[1], 1); mbar_init(&xready[0], 16); mbar_init(&xready[1], 16);
        for (int i = 0; i < 4; ++i) mbar_init(&xfree[i], 1);
        mbar_init(g_full, 1); mbar_init(g_empty, 8);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    cluster_sync_all();                                         // barriers of both CTAs initialised before anything remote
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();
    tcgen05_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);    // warp-uniform for the compiler

    if (warp == 0) {
        // ===================================================== TMA producer
        // Warp-uniform control flow; one elected lane issues the TMA instructions of a stage.
        {
            int stage = 0; uint32_t phase = 0, h0_phase = 0, g_phase = 0;
            long long t_wempty = 0;
            const uint32_t w_addr = smem_u32(sW);
            const uint32_t wfull_addr = smem_u32(w_full), wempty_addr = smem_u32(w_empty);
            for (int pt = pair0; pt < ptiles; pt += npairs) {
                const int tile = pt * 2 + (int)rank;
                if (p.h0_from_tma) {
                    mbar_wait(h0_empty, h0_phase ^ 1);
                    if (elect_one()) {   // own rows, but the arrival and the bytes go to the leader's barrier
                        mbar_expect_tx_cluster(mapa_rank0(smem_u32(h0_full)), H0_BYTES);
                        tma_load_2d_pair(smem_u32(sH0), &maps.m[0], smem_u32(h0_full), 0, tile * FBM);
                    }
                    __syncwarp();
                    h0_phase ^= 1;
                }
                for (int step = 0; step < nsteps; ++step) {
                    const int net = (sampler && (p.T - 1 - step) < p.K && !p.use_base_policy) ? 1 : 0;
                    for (int l = 0; l < p.nlayers; ++l) {
                        const Layer& L = p.L[net][l];
                        const int n_cur = L.n < 256 ? L.n : 256, nhc = L.n / n_cur;
                        const int kx = L.a_src >= 1 ? H / WKE : 0, kh = L.a_src != 1 ? 64 / WKE : 0;
                        const CUtensorMap* wm = &maps.m[L.wmap];
                        const int n_mine = n_cur / 2;                      // this CTA's share of the B tile's columns
                        const uint32_t tx = (uint32_t)(WKE * n_mine * 2);
                        const int nbox = n_mine / 64;
                        if (HASG && L.gate_load_map >= 0) {
                            // gate tile of this layer: needed by its epilogue only, so it rides ahead of the weights
                            mbar_wait(g_empty, g_phase ^ 1); g_phase ^= 1;
                            if (elect_one()) {
                                mbar_expect_tx(g_full, X_BYTES);
                                for (int kb = 0; kb < XT; ++kb) tma_load_2d(sG + kb * 16384, &maps.m[L.gate_load_map], g_full, kb * 64, tile * FBM);
                            }
                            __syncwarp();
                        }
                        for (int nh = 0; nh < nhc; ++nh) {
                            const int col = nh * n_cur + (int)rank * n_mine;
                            int krow = kx ? L.wrow_x : L.wrow_h0;
                            for (int s = 0; s < kx + kh; ++s) {
                                if (s == kx) krow = L.wrow_h0;
                                const uint32_t full_bar = wfull_addr + stage * 8;
                                if (TIMING) { const long long c0 = clock64(); mbar_wait_addr(wempty_addr + stage * 8, phase ^ 1); t_wempty += clock64() - c0; }
                                else mbar_wait_addr(wempty_addr + stage * 8, phase ^ 1);
                                if (elect_one()) {
                                    const uint32_t dst = w_addr + stage * STAGE_BYTES;
                                    mbar_expect_tx_cluster(mapa_rank0(full_bar), tx);
                                    for (int j = 0; j < nbox; ++j) tma_load_2d_pair(dst + j * (WKE * 128), wm, full_bar, col + j * 64, krow);
                                }
                                __syncwarp();
                                krow += WKE;
                                if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                            }
                        }
                    }
                }
            }
            if (TIMING && p.dbg && lane == 0) p.dbg[blockIdx.x * 8 + 0] = t_wempty;
        }
    } else if (warp == 1) {
        // ===================================================== MMA issuer
        // The issuing thread is latency bound on its own instruction stream (~6 cycles per dependent instruction,
        // measured with tools/mma_probe.py), so descriptors are kept as 32-bit halves: the high word and the B
        // descriptors of the four ring slots are loop invariants, the A descriptor advances by an add.
        {
            int stage = 0; uint32_t phase = 0, h0_phase = 0, xr_phase = 0;
            const uint32_t desc_hi = (1024u >> 4) | (1u << 14) | (2u << 29);          // SBO = 1024 B, version 1, SWIZZLE_128B
            const uint32_t a_lo_x = ((smem_u32(sX) >> 4) & 0x3FFFu) | (1u << 16);     // K-major A: LBO = 16 B
            const uint32_t a_lo_h0 = ((smem_u32(sH0) >> 4) & 0x3FFFu) | (1u << 16);
            const uint32_t b_lo_0 = ((smem_u32(sW) >> 4) & 0x3FFFu) | ((uint32_t)(WKE * 128 >> 4) << 16);  // MN-major B: LBO = one 64-column atom
            const uint32_t wfull_addr = smem_u32(w_full), wempty_addr = smem_u32(w_empty);
            constexpr int S_HALF = (XT / 2) * (64 / WKE);         // first ring stage that reads X tile XT/2
            long long t_x = 0, t_w = 0; const long long t_begin = TIMING ? clock64() : 0;
            for (int pt = pair0; pt < ptiles && rank == 0; pt += npairs) {
                bool h0_waited = false;
                for (int step = 0; step < nsteps; ++step) {
                    const int net = (sampler && (p.T - 1 - step) < p.K && !p.use_base_policy) ? 1 : 0;
                    for (int l = 0; l < p.nlayers; ++l) {
                        const Layer& L = p.L[net][l];
                        const int n_cur = L.n < 256 ? L.n : 256, nhc = L.n / n_cur;
                        const int kx = L.a_src >= 1 ? H / WKE : 0, kh = L.a_src != 1 ? 64 / WKE : 0;
                        const uint32_t idesc = make_idesc(FBM * 2, n_cur, false, true);
                        const bool h0_rel = L.h0_last && p.h0_from_tma;
                        // xready[0]: the previous epilogue wrote X tiles [0, XT/2) (or H0) and drained the first accumulator half;
                        // xready[1]: tiles [XT/2, XT) and the second half.  The second wait is deferred to the first stage that needs it.
                        if (TIMING) { const long long c0 = clock64(); mbar_wait(&xready[0], xr_phase); t_x += clock64() - c0; } else mbar_wait(&xready[0], xr_phase);
                        bool xr1_waited = false;
                        if (kx == 0) { mbar_wait(&xready[1], xr_phase); xr1_waited = true; }
                        if (L.a_src != 1 && p.h0_from_tma && !h0_waited) { mbar_wait(h0_full, h0_phase); h0_phase ^= 1; h0_waited = true; }
                        tcgen05_fence_after();
                        for (int nh = 0; nh < nhc; ++nh) {
                            const uint32_t tmem_d = tmem_base + (uint32_t)(nh * 256);
                            const bool last_half_of_two = (nhc == 2 && nh == 1);
                            uint32_t accf = 0u;
                            uint32_t a_lo = kx ? a_lo_x : a_lo_h0;
                            if (last_half_of_two && kx == 0) {            // this layer never reads X: the epilogue may overwrite it at once
                                if (elect_one()) { for (int j = 0; j < XT / 2; ++j) tcgen05_commit_pair(smem_u32(&xfree[j])); }
                                __syncwarp();
                            }
                            for (int s = 0; s < kx + kh; ++s) {
                                if (s == kx) a_lo = a_lo_h0;
                                if (!xr1_waited && s == S_HALF) {
                                    if (TIMING) { const long long c0 = clock64(); mbar_wait(&xready[1], xr_phase); t_x += clock64() - c0; } else mbar_wait(&xready[1], xr_phase);
                                    xr1_waited = true;
                                }
                                if (TIMING) { const long long c0 = clock64(); mbar_wait_addr(wfull_addr + stage * 8, phase); t_w += clock64() - c0; }
                                else mbar_wait_addr(wfull_addr + stage * 8, phase);
                                tcgen05_fence_after();
                                const uint32_t b_lo = b_lo_0 + (uint32_t)stage * (STAGE_BYTES >> 4);
                                // the stage that finishes X tile j (j < XT/2) in the last n-half frees it for the epilogue
                                const bool free_tile = last_half_of_two && s < S_HALF && s < kx;
                                if (elect_one()) {
                                    umma_bf16_split_pair(tmem_d, a_lo, b_lo, desc_hi, idesc, accf);
                                    umma_bf16_split_pair(tmem_d, a_lo + 2u, b_lo + (2048u >> 4), desc_hi, idesc, 1u);
                                    umma_bf16_split_pair(tmem_d, a_lo + 4u, b_lo + (4096u >> 4), desc_hi, idesc, 1u);
                                    umma_bf16_split_pair(tmem_d, a_lo + 6u, b_lo + (6144u >> 4), desc_hi, idesc, 1u);
                                    tcgen05_commit_pair(wempty_addr + stage * 8);
                                    if (free_tile) tcgen05_commit_pair(smem_u32(&xfree[s]));
                                }
                                __syncwarp();
                                accf = 1u;
                                a_lo += (16384u >> 4);                            // next 64-column tile of A
                                if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                            }
                            if (elect_one()) tcgen05_commit_pair(smem_u32(&acc_full[nh]));
                            __syncwarp();
                        }
                        if (!xr1_waited) mbar_wait(&xready[1], xr_phase);
                        xr_phase ^= 1;
                        if (h0_rel) { if (elect_one()) tcgen05_commit_pair(smem_u32(h0_empty)); __syncwarp(); }
                    }
                }
            }
            if (TIMING && p.dbg && lane == 0) { p.dbg[blockIdx.x * 8 + 1] = t_x; p.dbg[blockIdx.x * 8 + 2] = t_w; p.dbg[blockIdx.x * 8 + 3] = clock64() - t_begin; }
        }
    } else {
        // ===================================================== epilogue warps (8: two per TMEM lane quadrant)
        const int quad = warp & 3;                               // TMEM lane quadrant this warp may access
        const int half = (warp - 2) >> 2;                        // 0: first half of the columns, 1: second half
        const int rloc = quad * 32 + lane;                       // row inside the tile == TMEM lane
        const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
        const uint32_t x_addr = smem_u32(sX), h0_addr = smem_u32(sH0), g_addr = smem_u32(sG);
        const bool store_thread = (warp == 2 && lane == 0);
        uint32_t gfull_phase = 0;
        // xready lives in the leader CTA: its MMA warp needs both CTAs' epilogues
        const uint32_t xr0 = mapa_rank0(smem_u32(&xready[0]));
        const uint32_t xr1 = mapa_rank0(smem_u32(&xready[1]));
        const int etid = threadIdx.x - 64;                       // 0..255
        uint32_t acc_phase[2] = {0u, 0u}, xf_phase = 0u;
        int bias_buf = 0;
        const int A = p.A;
        float x[16];                                             // sampler: this thread's half of the row's x
#pragma unroll
        for (int a = 0; a < 16; ++a) x[a] = 0.f;
        bool first = true;
        float csum[2][2] = {};                                   // column sums: thread etid (< H/2) owns columns 2*etid, 2*etid+1
        long long t_acc = 0, t_gen = 0, t_fin = 0;
        for (int pt = pair0; pt < ptiles; pt += npairs) {
            const int tile = pt * 2 + (int)rank;
            const int row = tile * FBM + rloc;
            const bool valid = row < p.rows;
            const float* obs_row = p.obs + (size_t)(valid ? row : 0) * p.Do;
            if (sampler) {
                // tile prologue: x_T (injected or Philox slot 0), first H0 image
#pragma unroll
                for (int b4 = 0; b4 < 4; ++b4) {
                    float nz[4] = {0.f, 0.f, 0.f, 0.f};
                    const int a0 = half * 16 + b4 * 4;
                    if (valid && a0 < A && !p.xT) philox_normal4(p.seed, p.offset, p.row_offset + row, 0, a0 >> 2, nz);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int a = a0 + e;
                        float v = 0.f;
                        if (valid && a < A) {
                            v = p.xT ? p.xT[(size_t)row * A + a] : nz[e];
                            if (p.chains_out && p.K == p.T) p.chains_out[((size_t)row * (p.K + 1)) * A + a] = v;
                        }
                        x[b4 * 4 + e] = v;
                    }
                }
                build_h0_half(h0_addr, rloc, half, x, obs_row, A, p.Do, p.T, p.T - 1, valid);
                fence_async_smem();
                __syncwarp();
                if (lane == 0) { mbar_arrive_cluster(xr0); mbar_arrive_cluster(xr1); }
            } else if (first) {
                if (lane == 0) { mbar_arrive_cluster(xr0); mbar_arrive_cluster(xr1); }   // "TMEM is free" for the very first layer
            }
            first = false;
            for (int step = 0; step < nsteps; ++step) {
                const int t_s = p.T - 1 - step;
                const int net = (sampler && t_s < p.K && !p.use_base_policy) ? 1 : 0;
                for (int l = 0; l < p.nlayers; ++l) {
                    const Layer& L = p.L[net][l];
                    const bool final_layer = (l == p.nlayers - 1) && p.final_mode != FINAL_STORE;
                    // stage this layer's bias in shared memory while the MMAs run (double buffered across layers)
                    float* sb = sBias + bias_buf * 512; bias_buf ^= 1;
                    if (L.bias) { for (int i = etid; i < (final_layer ? A : L.n); i += 256) sb[i] = __ldg(L.bias + i); }
                    long long c_epi = TIMING ? clock64() : 0;
                    if (!final_layer) {
                        // ---------------- generic layer: TMEM -> X (in place).  A 512-wide layer is drained in two phases:
                        // columns [0,256) as soon as the first n-half's MMAs are done - while the second half's MMAs still run
                        // (X tile j is overwritten only after those MMAs have consumed it: xfree[j]) - then columns [256,512).
                        // The next layer's MMAs start on X tiles [0, XT/2) while phase two is still writing the rest.
                        const bool two_half = (L.n > 256);
                        const int nphase = two_half ? 2 : 1;
                        const uint32_t* min_row = L.mask_in ? L.mask_in + (size_t)row * (H / 32) : nullptr;
                        uint32_t* mout_row = L.mask_out ? L.mask_out + (size_t)row * (H / 32) : nullptr;
                        const bool gate_in = HASG && L.gate_load_map >= 0;
                        const bool mish = HASG && L.act == 2;
                        for (int hph = 0; hph < nphase; ++hph) {
                            mbar_wait(&acc_full[hph], acc_phase[hph]); acc_phase[hph] ^= 1;
                            if (TIMING) { const long long c1 = clock64(); t_acc += c1 - c_epi; c_epi = c1; }
                            tcgen05_fence_after();
                            if (hph == 0) {
                                if (store_thread) tma_store_wait_read();   // earlier TMA stores must have finished reading X
                                epi_barrier();                             // ... and every warp is done with the previous layer (bias / colsum)
                                if (gate_in) { mbar_wait(g_full, gfull_phase); gfull_phase ^= 1; }
                            }
                            constexpr int nch = 4;                         // 32-column chunks per warp and phase
                            const int c_first = hph * 8 + half * nch;
                            if (mish) {
                                // Mish layers (critic forward): a ROLLED loop over groups of 8 columns.  The unrolled 4 x 32-column
                                // body below is ~45 KB of SASS per phase for this mode and the epilogue warps spent 2.4 x as many
                                // cycles waiting for instruction fetch as issuing (ncu source page); this body stays cache resident.
                                const uint32_t t0 = tmem_base + lane_base + (uint32_t)(c_first * 32);
                                const uint32_t row_off = (uint32_t)rloc * 128u, sw = (uint32_t)(rloc & 7);
                                const bool gstore = L.gate_store_map >= 0, hasb = L.bias != nullptr;
                                auto group8 = [&](const uint32_t (&r)[8], const int col0) {
                                    float v[8], gt[8];
#pragma unroll
                                    for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(r[j]);
                                    if (hasb) {
                                        const float4 b0 = *reinterpret_cast<const float4*>(sb + col0), b1 = *reinterpret_cast<const float4*>(sb + col0 + 4);
                                        v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w; v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
                                    }
#pragma unroll
                                    for (int j = 0; j < 8; ++j) { float y; mish_and_grad(v[j], y, gt[j]); v[j] = y; }
                                    const uint32_t off = (uint32_t)(col0 >> 6) * 16384u + row_off + (((uint32_t)((col0 & 63) >> 3) ^ sw) << 4);
                                    if (gstore) st_shared_v4(g_addr + off, pack_bf16(gt[0], gt[1]), pack_bf16(gt[2], gt[3]), pack_bf16(gt[4], gt[5]), pack_bf16(gt[6], gt[7]));
                                    st_shared_v4(x_addr + off, pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
                                };
                                uint32_t ra8[8], rb8[8];
                                tmem_ld8_async(t0, ra8);
#pragma unroll 1
                                for (int g2 = 0; g2 < nch * 4; g2 += 2) {
                                    tmem_ld_wait8(ra8);
                                    tmem_ld8_async(t0 + (uint32_t)((g2 + 1) * 8), rb8);
                                    group8(ra8, c_first * 32 + g2 * 8);
                                    tmem_ld_wait8(rb8);
                                    if (g2 + 2 < nch * 4) tmem_ld8_async(t0 + (uint32_t)((g2 + 2) * 8), ra8);
                                    group8(rb8, c_first * 32 + (g2 + 1) * 8);
                                }
                            } else {
                            if constexpr (H == 512) {
                            // H = 512 keeps the fully unrolled chunk loop: rolling it costs register spills there and measured slower
                            uint32_t mo[4] = {0u, 0u, 0u, 0u};
                            uint4 mi4 = make_uint4(0u, 0u, 0u, 0u);
                            uint32_t ra[32], rb[32];
                            tmem_ld32_async(tmem_base + lane_base + (uint32_t)(c_first * 32), ra);
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int c = c_first + u;
                                uint32_t (&r)[32] = (u & 1) ? rb : ra;
                                tmem_ld_wait(r);
                                if (u < 3) tmem_ld32_async(tmem_base + lane_base + (uint32_t)((c + 1) * 32), (u & 1) ? ra : rb);
                                const int n0 = c * 32;
                                float v[32];
#pragma unroll
                                for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
                                if (L.bias) {
#pragma unroll
                                    for (int j = 0; j < 32; j += 4) {
                                        const float4 b4 = *reinterpret_cast<const float4*>(sb + n0 + j);
                                        v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
                                    }
                                }
                                if (L.act == 1) {
                                    if (mout_row) {
                                        uint32_t bits = 0u;
#pragma unroll
                                        for (int j = 0; j < 32; ++j) bits |= (v[j] > 0.f ? 1u : 0u) << j;
                                        mo[u] = bits;
                                        if (u == 3 && valid) *reinterpret_cast<uint4*>(mout_row + (c - 3)) = make_uint4(mo[0], mo[1], mo[2], mo[3]);
                                    }
#pragma unroll
                                    for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
                                }
                                const uint32_t toff = (uint32_t)(n0 >> 6) * 16384u + (uint32_t)rloc * 128u;
                                const int cbg = (n0 & 63) >> 3;
                                if (gate_in) {
#pragma unroll
                                    for (int q = 0; q < 4; ++q) {
                                        uint32_t gw[4];
                                        ld_shared_v4(g_addr + toff + (uint32_t)(((cbg + q) ^ (rloc & 7)) << 4), gw[0], gw[1], gw[2], gw[3]);
#pragma unroll
                                        for (int e = 0; e < 4; ++e) {
                                            const float2 gf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&gw[e]));
                                            v[q * 8 + e * 2] *= gf.x; v[q * 8 + e * 2 + 1] *= gf.y;
                                        }
                                    }
                                }
                                if (min_row) {
                                    if (u == 0) mi4 = valid ? *reinterpret_cast<const uint4*>(min_row + c) : make_uint4(0u, 0u, 0u, 0u);
                                    const uint32_t bits = u == 0 ? mi4.x : (u == 1 ? mi4.y : (u == 2 ? mi4.z : mi4.w));
#pragma unroll
                                    for (int j = 0; j < 32; ++j) v[j] = ((bits >> j) & 1u) ? v[j] : 0.f;
                                }
                                // first phase of a two-phase layer: the second n-half's MMAs must be done with X tile c/2
                                if (two_half && hph == 0 && (u & 1) == 0) mbar_wait(&xfree[c >> 1], xf_phase);
#pragma unroll
                                for (int q = 0; q < 4; ++q)
                                    st_shared_v4(x_addr + toff + (uint32_t)(((cbg + q) ^ (rloc & 7)) << 4),
                                                 pack_bf16(v[q * 8 + 0], v[q * 8 + 1]), pack_bf16(v[q * 8 + 2], v[q * 8 + 3]),
                                                 pack_bf16(v[q * 8 + 4], v[q * 8 + 5]), pack_bf16(v[q * 8 + 6], v[q * 8 + 7]));
                            }
                            } else {
                            uint32_t ra[32], rb[32];
                            tmem_ld32_async(tmem_base + lane_base + (uint32_t)(c_first * 32), ra);
                            // one 32-column chunk: TMEM registers -> (+bias, ReLU (+mask out), x gate, x mask in) -> bf16 -> X
                            auto chunk = [&](const uint32_t (&r)[32], const int c, const bool first_of_pair, const uint32_t mask_in_bits, uint32_t& mask_out_bits) {
                                const int n0 = c * 32;
                                float v[32];
#pragma unroll
                                for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
                                if (L.bias) {
#pragma unroll
                                    for (int j = 0; j < 32; j += 4) {
                                        const float4 b4 = *reinterpret_cast<const float4*>(sb + n0 + j);
                                        v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
                                    }
                                }
                                if (L.act == 1) {
                                    if (mout_row) {
                                        uint32_t bits = 0u;
#pragma unroll
                                        for (int j = 0; j < 32; ++j) bits |= (v[j] > 0.f ? 1u : 0u) << j;
                                        mask_out_bits = bits;
                                    }
#pragma unroll
                                    for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
                                }
                                const uint32_t toff = (uint32_t)(n0 >> 6) * 16384u + (uint32_t)rloc * 128u;
                                const int cbg = (n0 & 63) >> 3;
                                if (gate_in) {
#pragma unroll
                                    for (int q = 0; q < 4; ++q) {
                                        uint32_t gw[4];
                                        ld_shared_v4(g_addr + toff + (uint32_t)(((cbg + q) ^ (rloc & 7)) << 4), gw[0], gw[1], gw[2], gw[3]);
#pragma unroll
                                        for (int e = 0; e < 4; ++e) {
                                            const float2 gf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&gw[e]));
                                            v[q * 8 + e * 2] *= gf.x; v[q * 8 + e * 2 + 1] *= gf.y;
                                        }
                                    }
                                }
                                if (min_row) {
#pragma unroll
                                    for (int j = 0; j < 32; ++j) v[j] = ((mask_in_bits >> j) & 1u) ? v[j] : 0.f;
                                }
                                // first phase of a two-phase layer: the second n-half's MMAs must be done with X tile c/2
                                if (two_half && hph == 0 && first_of_pair) mbar_wait(&xfree[c >> 1], xf_phase);
#pragma unroll
                                for (int q = 0; q < 4; ++q)
                                    st_shared_v4(x_addr + toff + (uint32_t)(((cbg + q) ^ (rloc & 7)) << 4),
                                                 pack_bf16(v[q * 8 + 0], v[q * 8 + 1]), pack_bf16(v[q * 8 + 2], v[q * 8 + 3]),
                                                 pack_bf16(v[q * 8 + 4], v[q * 8 + 5]), pack_bf16(v[q * 8 + 6], v[q * 8 + 7]));
                            };
                            // ROLLED over chunk pairs (the two TMEM register buffers alternate inside one iteration): half the SASS of the
                            // 4 x unrolled form - the epilogue warps were stalling on instruction fetch more often than they issued
                            auto chunk_pair = [&](const int up) {
                                const int c = c_first + up;
                                uint2 mi2 = make_uint2(0u, 0u), mo2 = make_uint2(0u, 0u);
                                if (min_row && valid) mi2 = *reinterpret_cast<const uint2*>(min_row + c);
                                tmem_ld_wait(ra);
                                tmem_ld32_async(tmem_base + lane_base + (uint32_t)((c + 1) * 32), rb);
                                chunk(ra, c, true, mi2.x, mo2.x);
                                tmem_ld_wait(rb);
                                if (up + 2 < nch) tmem_ld32_async(tmem_base + lane_base + (uint32_t)((c + 2) * 32), ra);
                                chunk(rb, c + 1, false, mi2.y, mo2.y);
                                if (mout_row && L.act == 1 && valid) *reinterpret_cast<uint2*>(mout_row + c) = mo2;
                            };
#pragma unroll 1
                            for (int up = 0; up < nch; up += 2) chunk_pair(up);
                            }
                            }
                            tcgen05_fence_before();
                            fence_async_smem();
                            if (gate_in) { __syncwarp(); if (lane == 0) mbar_arrive(g_empty); }
                            epi_barrier();
                            if (store_thread && (L.store_map >= 0 || (mish && L.gate_store_map >= 0))) {
                                const int kb0 = two_half ? hph * (XT / 2) : 0, kb1 = two_half ? kb0 + XT / 2 : L.n / 64;
                                if (L.store_map >= 0)
                                    for (int kb = kb0; kb < kb1; ++kb) tma_store_2d(&maps.m[L.store_map], sX + kb * 16384, kb * 64, tile * FBM);
                                if (mish && L.gate_store_map >= 0)
                                    for (int kb = kb0; kb < kb1; ++kb) tma_store_2d(&maps.m[L.gate_store_map], sG + kb * 16384, kb * 64, tile * FBM);
                                tma_store_commit();
                            }
                            __syncwarp();
                            if (lane == 0) { mbar_arrive_cluster((two_half && hph == 1) ? xr1 : xr0); if (!two_half) mbar_arrive_cluster(xr1); }
                        }
                        if (two_half) xf_phase ^= 1;
                        if (L.colsum_slot >= 0) {
                            // bias gradient: column sums of the bf16 tile just written (valid rows only).  Runs while the
                            // next layer's MMAs already read X; the next epilogue's barrier orders it before X is rewritten.
                            const int nrows = max(0, min(FBM, p.rows - tile * FBM));
                            if (etid < H / 2) {
                                const int kb = etid >> 5, w = etid & 31;
                                const uint32_t base = x_addr + (uint32_t)kb * 16384u + (uint32_t)(w & 3) * 4u;
                                float s0 = 0.f, s1 = 0.f;
                                for (int r = 0; r < nrows; ++r) {
                                    uint32_t word;
                                    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(word) : "r"(base + (uint32_t)r * 128u + (uint32_t)(((w >> 2) ^ (r & 7)) << 4)));
                                    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&word));
                                    s0 += f.x; s1 += f.y;
                                }
                                if (L.colsum_slot == 0) { csum[0][0] += s0; csum[0][1] += s1; } else { csum[1][0] += s0; csum[1][1] += s1; }
                            }
                        }
                        if (TIMING) t_gen += clock64() - c_epi;
                    } else {
                        // ---------------- final layer: eps of this row sits in TMEM columns [0, 32); each half takes 16
                        mbar_wait(&acc_full[0], acc_phase[0]); acc_phase[0] ^= 1;
                        if (TIMING) { const long long c1 = clock64(); t_acc += c1 - c_epi; c_epi = c1; }
                        tcgen05_fence_after();
                        uint32_t r[16];
                        tmem_ld16(tmem_base + lane_base + (uint32_t)(half * 16), r);
                        tcgen05_fence_before();
                        // eps / log-prob modes touch neither X nor H0 from here on: hand TMEM back before the math
                        if (!sampler) { __syncwarp(); if (lane == 0) { mbar_arrive_cluster(xr0); mbar_arrive_cluster(xr1); } }
                        epi_barrier();                                  // sb (bias) visible
                        const int abase = half * 16;
                        float eps[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) eps[j] = __uint_as_float(r[j]) + ((L.bias && abase + j < A) ? sb[abase + j] : 0.f);
                        if (p.final_mode == FINAL_EPS) {
                            if (valid) {
#pragma unroll
                                for (int j = 0; j < 16; ++j) if (abase + j < A) p.out[(size_t)row * A + abase + j] = eps[j];
                            }
                        } else if (p.final_mode == FINAL_LOGP) {
                            if (valid) {
                                const float *pv, *nx; int t;
                                if (p.chains) {
                                    const int b = row / p.K, k = row % p.K;
                                    pv = p.chains + ((size_t)b * (p.K + 1) + k) * A; nx = pv + A; t = p.K - 1 - k;
                                } else { pv = p.prev + (size_t)row * A; nx = p.next + (size_t)row * A; t = p.trow[row]; }
                                float xv[16], nv[16];
#pragma unroll
                                for (int j = 0; j < 16; ++j) { const bool ok = abase + j < A; xv[j] = ok ? __ldg(pv + abase + j) : 0.f; nv[j] = ok ? __ldg(nx + abase + j) : 0.f; }
                                const StepConst sc = step_const(p.sch, p.T, t);
                                const float sd = logprob_std(sc, p.min_lp_std);
                                const float lgs = 0.91893853320467274f + logf(sd);
#pragma unroll
                                for (int j = 0; j < 16; ++j) if (abase + j < A)
                                    p.out[(size_t)row * A + abase + j] = logprob_elem_c(xv[j], eps[j], nv[j], sc, sd, lgs, p.dcv, nullptr, nullptr);
                            }
                        } else {   // FINAL_SAMPLE: posterior mean, clipped noise, x update (diffusion_vpg.py:198-206,239-243,301-338)
                            const StepConst sc = step_const(p.sch, p.T, t_s);
                            const float sd = sample_std(sc, t_s, p.hp);
                            if (valid) {
#pragma unroll
                                for (int b4 = 0; b4 < 4; ++b4) {
                                    const int a0 = abase + b4 * 4;
                                    if (a0 < A) {
                                        float nz[4];
                                        if (p.noise) {
#pragma unroll
                                            for (int e = 0; e < 4; ++e) nz[e] = (a0 + e < A) ? __ldg(p.noise + ((size_t)step * p.rows + row) * A + a0 + e) : 0.f;
                                        } else philox_normal4(p.seed, p.offset, p.row_offset + row, 1 + step, a0 >> 2, nz);
#pragma unroll
                                        for (int e = 0; e < 4; ++e) {
                                            const int a = a0 + e;
                                            if (a < A) {
                                                const float xn = ddpm_step_elem_c(x[b4 * 4 + e], eps[b4 * 4 + e], nz[e], sc, sd, p.hp, t_s == 0);
                                                x[b4 * 4 + e] = xn;
                                                if (p.chains_out && t_s <= p.K) p.chains_out[((size_t)row * (p.K + 1) + (p.K - t_s)) * A + a] = xn;
                                                if (t_s == 0) p.actions[(size_t)row * A + a] = xn;
                                            }
                                        }
                                    }
                                }
                            }
                            if (step + 1 < nsteps) {
                                build_h0_half(h0_addr, rloc, half, x, obs_row, A, p.Do, p.T, t_s - 1, valid);
                                fence_async_smem();
                            }
                        }
                        __syncwarp();
                        // the sampler's last step hands over to the next tile's prologue instead
                        if (lane == 0 && sampler && step + 1 < nsteps) { mbar_arrive_cluster(xr0); mbar_arrive_cluster(xr1); }
                        if (TIMING) t_fin += clock64() - c_epi;
                    }
                }
            }
        }
        if (store_thread) tma_store_wait_all();
        if (p.colsum_part && etid < H / 2) {
            float* dst = p.colsum_part + (size_t)blockIdx.x * 2 * H + 2 * etid;
            dst[0] = csum[0][0]; dst[1] = csum[0][1]; dst[H] = csum[1][0]; dst[H + 1] = csum[1][1];
        }
        if (TIMING && p.dbg && warp == 2 && lane == 0) { p.dbg[blockIdx.x * 8 + 4] = t_acc; p.dbg[blockIdx.x * 8 + 5] = t_gen; p.dbg[blockIdx.x * 8 + 6] = t_fin; }
    }
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();                     // the peer may still be signalling our barriers / reading our B halves
    if (warp == 1) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ------------------------------------------------------------------ host side
// weight operand [K][N] bf16 row-major (leading dimension ld): box [2 WK k][64 n]
static int weight_map(CUtensorMap* m, const void* base, uint64_t K, uint64_t N, uint64_t ld) { return make_map(m, base, K, N, ld, WK * 2, 64); }
// row tile source / destination [rows][cols] bf16 row-major: box [128 rows][64 cols]
static int rowtile_map(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols) { return make_map(m, base, rows, cols, cols, FBM, 64); }

// number of CTAs a chain launch uses (CTA pairs: an even grid)
static int chain_grid(const dppo_handle* h, int rows) {
    const int ntiles = (rows + FBM - 1) / FBM;
    const int pairs = (ntiles + 1) / 2, maxp = h->sm_count / 2;
    return 2 * (pairs < maxp ? pairs : maxp);
}

template <int H>
static int launch_chain_t(dppo_handle* h, cudaStream_t s, const Maps& maps, const Params& p, double flops) {
    auto kern = p.dbg ? chain_kernel<H, true> : chain_kernel<H, false>;
    static bool attr_set_dev[64] = {};      // function attributes are per device
    bool& attr_set = attr_set_dev[h->device & 63];
    if (!attr_set) {
        CUDA_TRY(cudaFuncSetAttribute(chain_kernel<H, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)chain_smem_bytes<H>()));
        CUDA_TRY(cudaFuncSetAttribute(chain_kernel<H, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)chain_smem_bytes<H>()));
        attr_set = true;
    }
    const int grid = chain_grid(h, p.rows);
    prof_begin(h, s);
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1; cfg.blockDim = dim3(FTHREADS); cfg.gridDim = dim3(grid); cfg.dynamicSmemBytes = chain_smem_bytes<H>(); cfg.stream = s;
    cudaError_t le = cudaLaunchKernelEx(&cfg, kern, maps, p);
    if (le != cudaSuccess) DPPO_FAIL(-3, "fused chain (CTA pair) launch failed: %s", cudaGetErrorString(le));
    prof_end(h, s, flops, H == 512 ? 0 : 3);      // the two instantiations are different kernels: time them separately
    h->launches++; h->tc_launches++; h->fused_launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) DPPO_FAIL(-3, "fused chain launch failed: %s", cudaGetErrorString(e));
    return 0;
}
static int launch_chain(dppo_handle* h, cudaStream_t s, int H, const Maps& maps, const Params& p, double flops) {
    if (H == 512) return launch_chain_t<512>(h, s, maps, p, flops);
    if (H == 256) return launch_chain_t<256>(h, s, maps, p, flops);
    DPPO_FAIL(-7, "fused chain: unsupported hidden width %d", H);
}

}  // namespace fc

// ------------------------------------------------------------------ dev probe (tools/mma_probe.py)
// mode 0: the chain kernel's MMA issue sequence (poll a ready mbarrier, 2 x tcgen05.mma 128 x N x 16, commit) on
//         fixed operands: cycles per 2-MMA stage, i.e. the issue cost with no data dependence at all.
// mode 1: TMA round trip: one 16 KB weight stage (4 boxes from 4 lanes) at a time, issue -> mbarrier completion.
// mode 2: TMA throughput with `depth` stages in flight (depth <= 4), same lean producer loop as the chain kernel.
namespace fc {
__global__ void __launch_bounds__(128, 1) mma_probe_kernel(const __grid_constant__ CUtensorMap wmap, int mode, int iters, int N, int depth,
                                                           long long* out) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* sA = smem;                 // 16 KB
    uint8_t* sB = smem + 16384;         // 4 x 16 KB
    uint64_t* bars = (uint64_t*)(sB + 4 * 16384);
    uint64_t* done = bars; uint64_t* sink = bars + 1; uint64_t* tfull = bars + 2; uint64_t* ready = bars + 6;
    uint32_t* tmem_slot = (uint32_t*)(bars + 12);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < (16384 * 5) / 4; i += blockDim.x) ((uint32_t*)smem)[i] = 0x3c003c00u;
    if (threadIdx.x == 0) {
        mbar_init(done, 1); mbar_init(sink, 1); mbar_init(ready, 1);
        for (int i = 0; i < 4; ++i) mbar_init(&tfull[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (mode == 0 && warp == 1 && lane == 0) {
        const uint32_t idesc = make_idesc(128, N, false, true);
        const uint32_t desc_hi = (1024u >> 4) | (1u << 14) | (2u << 29);
        const uint32_t a_lo0 = ((smem_u32(sA) >> 4) & 0x3FFFu) | (1u << 16);
        const uint32_t b_lo_0 = ((smem_u32(sB) >> 4) & 0x3FFFu) | ((uint32_t)(WK * 128 >> 4) << 16);
        const uint32_t ready_addr = smem_u32(ready), sink_addr = smem_u32(sink);
        int stage = 0; uint32_t phase = 0; uint32_t a_lo = a_lo0;
        const long long t0 = clock64();
        // depth bits: 1 = commit per stage, 2 = poll a ready mbarrier per stage, 4 = tcgen05.fence::after per stage, 8 = 4 MMAs per stage
        const int nm = (depth & 8) ? 4 : 2;
        const uint32_t d1 = (depth & 16) ? tmem_base + 256u : tmem_base;     // bit 16: alternate between two accumulators
        for (int s = 0; s < iters; ++s) {
            if (depth & 2) mbar_wait_addr(ready_addr, 1);           // never arrived on: the parity-1 wait succeeds at once
            if (depth & 4) tcgen05_fence_after();
            const uint32_t b_lo = b_lo_0 + (uint32_t)stage * (STAGE_BYTES >> 4);
            umma_bf16_split(tmem_base, a_lo, b_lo, desc_hi, idesc, 1u);
            umma_bf16_split(d1, a_lo + 2u, b_lo + (2048u >> 4), desc_hi, idesc, 1u);
            if (nm == 4) {
                umma_bf16_split(tmem_base, a_lo, b_lo, desc_hi, idesc, 1u);
                umma_bf16_split(d1, a_lo + 2u, b_lo + (2048u >> 4), desc_hi, idesc, 1u);
            }
            if (depth & 1) tcgen05_commit_addr(sink_addr);
            a_lo = (s & 1) ? a_lo0 : a_lo + 4u;
            if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
        }
        const long long t1 = clock64();
        tcgen05_commit(done);
        mbar_wait(done, 0);
        const long long t2 = clock64();
        out[blockIdx.x * 2] = t1 - t0; out[blockIdx.x * 2 + 1] = t2 - t0;
    }
    if (mode >= 1 && warp == 0 && lane < 4) {
        const uint32_t w_addr = smem_u32(sB) + (uint32_t)lane * (WK * 128);
        const uint32_t tfull_addr = smem_u32(tfull);
        uint32_t ph[4] = {0, 0, 0, 0};
        const int D = mode == 1 ? 1 : depth;
        const long long t0 = clock64();
        int krow = (blockIdx.x * 32) % 512;
        for (int i = 0; i < D; ++i) {
            if (lane == 0) mbar_expect_tx_addr(tfull_addr + i * 8, 16384);
            __syncwarp(0xf);
            tma_load_2d_addr(w_addr + i * STAGE_BYTES, &wmap, tfull_addr + i * 8, lane * 64, krow);
            krow = (krow + 32) & 511;
        }
        int i = 0;
        for (int it = 0; it < iters; ++it) {
            mbar_wait_addr(tfull_addr + i * 8, ph[i & 3]); ph[i & 3] ^= 1;
            if (lane == 0) mbar_expect_tx_addr(tfull_addr + i * 8, 16384);
            __syncwarp(0xf);
            tma_load_2d_addr(w_addr + i * STAGE_BYTES, &wmap, tfull_addr + i * 8, lane * 64 + ((it >> 4) & 1) * 256, krow);
            krow = (krow + 32) & 511;
            if (++i == D) i = 0;
        }
        for (int k = 0; k < D; ++k) mbar_wait_addr(tfull_addr + k * 8, ph[k]);
        if (lane == 0) { out[blockIdx.x * 2] = clock64() - t0; out[blockIdx.x * 2 + 1] = iters + D; }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}
}  // namespace fc
