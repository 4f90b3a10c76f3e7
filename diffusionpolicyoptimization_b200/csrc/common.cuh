// Shared declarations for libdppo_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>
#include <string>
#include <vector>
#include "../../include/dppo_b200.h"

// ------------------------------------------------------------------ errors
void dppo_set_error(const char* fmt, ...);
#define DPPO_FAIL(code, ...) do { dppo_set_error(__VA_ARGS__); return (code); } while (0)
#define CUDA_TRY(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { \
    dppo_set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, cudaGetErrorString(_e)); return -2; } } while (0)
#define DPPO_TRY(expr) do { int _r = (expr); if (_r != 0) return _r; } while (0)

enum { SCH_BETAS = 0, SCH_ACP, SCH_SQRT_ACP, SCH_SQRT_1M_ACP, SCH_SQRT_RECIP, SCH_SQRT_RECIPM1,
       SCH_LOGVAR, SCH_COEF1, SCH_COEF2, SCH_ROWS };

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// ------------------------------------------------------------------ device math
__device__ __forceinline__ float softplus_f(float x) {
    // tf.math.softplus: log(exp(x) + 1), evaluated stably
    return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x)));
}
__device__ __forceinline__ float mish_f(float x) { return x * tanhf(softplus_f(x)); }
__device__ __forceinline__ float mish_grad_f(float x) {
    float sp = softplus_f(x);
    float th = tanhf(sp);
    float sg = 1.f / (1.f + expf(-x));
    return th + x * (1.f - th * th) * sg;
}
template <int ACT> __device__ __forceinline__ float act_f(float x) {
    if (ACT == DPPO_ACT_RELU + 1) return fmaxf(x, 0.f);
    if (ACT == DPPO_ACT_MISH + 1) return mish_f(x);
    return x;
}
__device__ __forceinline__ float act_rt(float x, int act1) {   // act1 = 0 none, 1 relu, 2 mish
    return act1 == 1 ? fmaxf(x, 0.f) : (act1 == 2 ? mish_f(x) : x);
}
__device__ __forceinline__ float act_grad_rt(float x, int act1) {
    return act1 == 1 ? (x > 0.f ? 1.f : 0.f) : (act1 == 2 ? mish_grad_f(x) : 1.f);
}

// ------------------------------------------------------------------ Philox4x32-10 (counter based)
struct Philox4 { uint32_t x, y, z, w; };
__host__ __device__ __forceinline__ Philox4 philox4x32_10(Philox4 c, uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * c.x, p1 = (uint64_t)M1 * c.z;
        Philox4 n;
        n.x = (uint32_t)(p1 >> 32) ^ c.y ^ k0;
        n.y = (uint32_t)p1;
        n.z = (uint32_t)(p0 >> 32) ^ c.w ^ k1;
        n.w = (uint32_t)p0;
        c = n; k0 += W0; k1 += W1;
    }
    return c;
}
// The noise stream of this library: standard normal for (global row, slot, element a).
//   counter = (a>>2 | slot<<8, offset_lo, row_lo, row_hi), key = (seed_lo, seed_hi + offset_hi)
//   u = (bits + 0.5) * 2^-32;  (n0,n1) = sqrt(-2 ln u0) * (cos, sin)(2 pi u1); (n2,n3) from (u2,u3).
__device__ __forceinline__ float philox_normal(uint64_t seed, uint64_t offset, int64_t row, int slot, int a) {
    Philox4 c;
    c.x = (uint32_t)(a >> 2) | ((uint32_t)slot << 8);
    c.y = (uint32_t)offset;
    c.z = (uint32_t)(uint64_t)row;
    c.w = (uint32_t)((uint64_t)row >> 32);
    Philox4 r = philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32) + (uint32_t)(offset >> 32));
    uint32_t b0 = (a & 2) ? r.z : r.x, b1 = (a & 2) ? r.w : r.y;
    float u0 = ((float)b0 + 0.5f) * 2.3283064365386963e-10f;
    float u1 = ((float)b1 + 0.5f) * 2.3283064365386963e-10f;
    u0 = fminf(fmaxf(u0, 1.1754944e-38f), 0.99999994f);
    float rad = sqrtf(-2.f * logf(u0));
    float sn, cs;
    sincospif(2.f * u1, &sn, &cs);
    return (a & 1) ? rad * sn : rad * cs;
}
// the four normals of Philox block `blk` (elements a = 4*blk .. 4*blk+3): identical values to philox_normal
__device__ __forceinline__ void philox_normal4(uint64_t seed, uint64_t offset, int64_t row, int slot, int blk, float (&out)[4]) {
    Philox4 c;
    c.x = (uint32_t)blk | ((uint32_t)slot << 8);
    c.y = (uint32_t)offset;
    c.z = (uint32_t)(uint64_t)row;
    c.w = (uint32_t)((uint64_t)row >> 32);
    Philox4 r = philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32) + (uint32_t)(offset >> 32));
#pragma unroll
    for (int hlf = 0; hlf < 2; ++hlf) {
        const uint32_t b0 = hlf ? r.z : r.x, b1 = hlf ? r.w : r.y;
        float u0 = ((float)b0 + 0.5f) * 2.3283064365386963e-10f;
        float u1 = ((float)b1 + 0.5f) * 2.3283064365386963e-10f;
        u0 = fminf(fmaxf(u0, 1.1754944e-38f), 0.99999994f);
        float rad = sqrtf(-2.f * logf(u0));
        float sn, cs;
        sincospif(2.f * u1, &sn, &cs);
        out[hlf * 2 + 0] = rad * cs; out[hlf * 2 + 1] = rad * sn;
    }
}
__device__ __forceinline__ uint32_t philox_uint(uint64_t seed, uint64_t offset, int64_t row, int slot) {
    Philox4 c;
    c.x = ((uint32_t)slot << 8);
    c.y = (uint32_t)offset;
    c.z = (uint32_t)(uint64_t)row;
    c.w = (uint32_t)((uint64_t)row >> 32);
    Philox4 r = philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32) + (uint32_t)(offset >> 32));
    return r.x;
}

// ------------------------------------------------------------------ model geometry
struct ActorOff {   // offsets (floats) into one actor's flat parameter vector
    size_t tw1, tb1, tw2, tb2, win, bin, w1, b1, w2, b2, w3, b3, n;
};
struct CriticOff { size_t win, bin, w1, b1, w2, b2, w3, b3, n; };

struct Geom {
    int Do, A, T, K, td, H, Hc, Din, KP, KPc;
    ActorOff ao; CriticOff co;
};

// derived, recomputed after every weight change of that net
// programmatic dependent launch for the short kernels at the end of an update: launch_pdl lets the kernel start while the previous
// kernel of the stream drains (hiding the launch gap); such a kernel calls pdl_grid_begin() before it touches global memory, which
// waits until the previous grids have completed and their writes are visible, then lets its own dependent launch early
__device__ __forceinline__ void pdl_grid_begin() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s; cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}

struct ActorDerived {
    float* sinemb;  // [T][td]
    float* thpre;   // [T][2td]
    float* temb;    // [T][td]
    float* bt;      // [T][H]   = b_in + temb(t) @ W_in[A:A+td]
    float* dte;     // [T][td] + a counter: scratch of the time-MLP backward (time_backward_body)
    float* w0p;     // [KP][H]  = rows of W_in for [x | obs], zero padded
    // no activation sits between block.l2 and the output layer: eps = (a1 W2 + b2 + u) W3 + b3 = a1 (W2 W3) + u W3 + (b2 W3 + b3).
    // Forward-only programs (the samplers, the log-prob forward) use the folded operands and skip the H x H product.
    float* w23;     // [H][A]   = W2 @ W3   (double accumulation, rounded once)
    float* b23;     // [A]      = b2 @ W3 + b3
};

struct OptState { float* m; float* v; int64_t step; size_t n; };

// A grow-only device buffer carved into 256-byte aligned slices by ws_take; ws_layout sizes it.  peak: the most bytes taken
// since the layout began (a nested program gives its slices back, see ws_room).
struct Workspace {
    char* base = nullptr; size_t cap = 0, used = 0, peak = 0;
};

struct dppo_handle {
    dppo_cfg cfg; int device; Geom g;
    int sm_count;
    float* params;        // [actor | actor_ft | critic | actor_ema]
    float* net_w[4];
    size_t net_n[4];
    ActorDerived ad[4];   // index by net id (critic entry: only w0p used = [KPc][Hc])
    float* sched;         // device [SCH_ROWS*T]
    float  sched_host[SCH_ROWS * 1024];
    OptState opt[2];
    float* grads;         // [nA + nC + 16]
    float* scalars;       // device scratch: [0..1] adv mean/std, [8..] metric sums
    Workspace ws;
    Workspace stage;      // device copies of the host arrays of the *_host calls
    cudaStream_t copy_stream = nullptr; cudaEvent_t copy_ev[9];   // chunked H2D / compute overlap of dppo_ppo_step_host
    // NCCL
    void* comm = nullptr; int rank = 0, world = 1;
    // peer-memory all-reduce fused with AdamW (dppo_comm_ipc_*): two alternating gradient buffers, flag barrier
    float* grads_buf[2] = {nullptr, nullptr}; int grads_cur = 0; float* gsum = nullptr; size_t grads_floats = 0;
    unsigned long long* flags = nullptr;             // [8] epoch written by each peer
    float* peer_grads[2][8] = {}; unsigned long long* peer_flags[8] = {}; int peers_attached = 0;
    unsigned long long epoch = 0;
    int* comm_status = nullptr;                      // device: raised by a peer barrier that timed out (lives in `scalars`)
    long long peer_timeout_cycles = 0;
    const int* skip_update = nullptr;                // device flag of the step in flight: non-zero = leave weights / moments untouched (bad minibatch indices)
    int64_t launches = 0;
    int64_t tc_launches = 0;
    int w0p_dirty[4] = {1, 1, 1, 1};  // ActorDerived::w0p is stale (rebuilt on demand by the FFMA layer-0 GEMM)
    int w23_dirty[4] = {1, 1, 1, 1};     // folded output-layer tables (ActorDerived::w23 / b23) need a rebuild
    int peer_two_shot = -1;           // DPPO_PEER_TWO_SHOT=0/1 (default: two-shot from 4 ranks)
    float* peer_gsum[8] = {nullptr};
    cudaStream_t aux_stream = nullptr; cudaEvent_t aux_ev[3] = {nullptr, nullptr, nullptr};
    float grad_clip_norm = 0.f;       // dppo_set_grad_clip_norm: per-variable tf.clip_by_norm before AdamW (<= 0: off)
    int deterministic = 0;            // DPPO_DETERMINISTIC=1: fixed-order split-K reductions instead of red.global.add
    int chain_dbg_idx = 0;
    long long* chain_dbg = nullptr;   // dev tool: per-CTA cycle counters of the last fused-chain launch [sm_count][8]
    int64_t fused_launches = 0;   // of those, fused layer-chain launches
    int cluster_max = -1; // max co-resident 16-CTA clusters (-1 unknown, 0 = not launchable)
    int last_path = 0;    // sampler path of the last dppo_sample: 1 cluster, 2 layered fp32, 3 tensor
    int force_path = 0;   // test hook: 0 auto, 1 force cluster sampler, 2 forbid it
    struct TcState* tc = nullptr;   // tcgen05 path state (tc_path.cuh)
    float* env_norm = nullptr;      // device [2 * obs_dim + 2 * action_dim]: obs_min, obs_max, action_min, action_max (dppo_set_env_normalization)
    struct TsState* ts = nullptr;   // split-precision tcgen05 path state (ts_path.cuh, DPPO_PREC_BF16X3)
    // live GEMM timing (dppo_profile_*): event pairs recorded around GEMM-class launches
    int prof_on = 0;
    std::vector<cudaEvent_t> prof_ev;   // pairs
    std::vector<int> prof_cls;          // kernel class of each pair: 0 fused chain <H = 512>, 1 tcgen05 GEMM, 2 FFMA SGEMM, 3 fused chain <H = 256>
    size_t prof_used = 0;
    double prof_flops[4] = {0, 0, 0, 0}, prof_ms_acc[4] = {0, 0, 0, 0}; int64_t prof_launches[4] = {0, 0, 0, 0};
    double prof_exec[4] = {0, 0, 0, 0};   // flops the tensor pipe executed (plane modes issue 3 or 6 products per algorithmic multiply-add)
};

// Every weight change of a net (set_weights, an applied PPO or pre-training step, ema_update, a skipped update) calls this: it marks
// every lazily rebuilt table of that net stale - w0p, w23 / b23 and the split-precision folded layers - so that the next reader
// rebuilds it.  The eagerly rebuilt copies (time tables, bf16 / plane operands) are rewritten by the same call that changed the
// weights.  A lazy table added later is listed here, once.
static void mark_weights_changed(dppo_handle* h, int net);

// profile bracket: call prof_begin before and prof_end after a GEMM-class launch
void prof_begin(dppo_handle* h, cudaStream_t s);
void prof_end(dppo_handle* h, cudaStream_t s, double flops, int cls, double exec_flops = -1.0);   // exec_flops: tensor-pipe flops actually issued (default: = flops)

// ------------------------------------------------------------------ workspace layout
// A program describes its buffers once, as a layout: a function that only takes slices (ws_take) and computes pointers from them.
// It launches nothing and reads nothing from the device.  ws_layout runs it twice: a counting pass whose high-water mark sizes
// the buffer, then the pass whose pointers the program uses.
template <typename T> static inline T* ws_take(Workspace& w, size_t count) {
    T* p = (T*)((uintptr_t)w.base + w.used);      // not dereferenced during the counting pass, where base may be stale
    w.used += (count * sizeof(T) + 255) / 256 * 256;
    if (w.used > w.peak) w.peak = w.used;
    return p;
}
template <typename T> static inline T* ws_take(dppo_handle* h, size_t count) { return ws_take<T>(h->ws, count); }
int ws_reserve(Workspace& w, size_t bytes, cudaStream_t s);   // grow-only; only ws_layout calls it
static inline int ws_check(const Workspace& w) {
    if (w.peak > w.cap) DPPO_FAIL(-7, "workspace layout takes %zu bytes, %zu reserved", w.peak, w.cap);
    return 0;
}
template <typename F> static int ws_layout(Workspace& w, cudaStream_t s, F&& layout) {
    w.used = w.peak = 0;
    layout();
    DPPO_TRY(ws_reserve(w, w.peak, s));
    w.used = w.peak = 0;
    layout();
    return ws_check(w);
}
// A nested program (tc_actor_forward, ts_actor_forward) appends its slices above the caller's at call time and gives them back when
// it returns; the caller holds pointers below w.used, so the buffer must not grow then.  The caller's layout makes room for it
// with ws_room (the nested layout counts towards peak, nothing stays taken); the nested program takes its slices with ws_append.
template <typename F> static void ws_room(Workspace& w, F&& layout) {
    const size_t mark = w.used;
    layout();
    w.used = mark;
}
template <typename F> static int ws_append(Workspace& w, F&& layout) {
    w.peak = w.used;
    layout();
    return ws_check(w);
}
