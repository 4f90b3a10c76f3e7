// libdppo_b200.so — C-ABI entry points (include/dppo_b200.h) and host-side orchestration.
#include "common.cuh"
#include "simt_kernels.cuh"
#include "sample_cluster.cuh"
#include "tc_path.cuh"
#include "ts_path.cuh"
#include <stdarg.h>
#include <dlfcn.h>
#include <cmath>

// ------------------------------------------------------------------ error plumbing
static thread_local char g_err[1024] = "";
void dppo_set_error(const char* fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}
extern "C" const char* dppo_last_error(void) { return g_err; }
extern "C" int dppo_abi_version(void) { return DPPO_ABI_VERSION; }
extern "C" size_t dppo_cfg_size(void) { return sizeof(dppo_cfg); }

#define KLAUNCH(h) do { (h)->launches++; } while (0)
#define KCHECK() do { cudaError_t _e = cudaGetLastError(); if (_e != cudaSuccess) { \
    dppo_set_error("kernel launch failed at %s:%d: %s", __FILE__, __LINE__, cudaGetErrorString(_e)); return -3; } } while (0)

extern "C" void dppo_cfg_default(dppo_cfg* c) {
    memset(c, 0, sizeof(*c));
    c->obs_dim = 11; c->action_dim = 3; c->horizon_steps = 4; c->cond_steps = 1;
    c->denoising_steps = 20; c->ft_denoising_steps = 10; c->time_dim = 16;
    c->actor_hidden = 512; c->critic_hidden = 256;
    c->actor_act = DPPO_ACT_RELU; c->critic_act = DPPO_ACT_MISH;
    c->precision = DPPO_PREC_FP32;
    c->denoised_clip_value = 1.0f; c->randn_clip_value = 3.0f; c->final_action_clip_value = -1.f;
    c->min_sampling_denoising_std = 0.1f; c->min_logprob_denoising_std = 0.1f;
    c->gamma_denoising = 0.99f; c->clip_ploss_coef = 0.01f; c->clip_ploss_coef_base = 0.01f; c->clip_ploss_coef_rate = 3.f;
    c->clip_vloss_coef = -1.f; c->norm_adv = 1; c->reward_horizon = 4; c->vf_coef = 0.5f;
    c->logprob_clip_lo = -5.f; c->logprob_clip_hi = 2.f;
    c->adam_beta1 = 0.9f; c->adam_beta2 = 0.999f; c->adam_eps = 1e-7f;
    c->weight_decay = 0.004f; c->pretrain_weight_decay = 1e-6f;
}

// ------------------------------------------------------------------ schedule (sampling.py:7-17, diffusion.py:58-73)
extern "C" int dppo_ddpm_schedule(int T, float* out) {
    if (T < 1 || T > 1024 || !out) DPPO_FAIL(-1, "dppo_ddpm_schedule: bad arguments (T=%d)", T);
    const double s = 0.008;
    const int steps = T + 1;
    std::vector<double> acp(steps);
    for (int i = 0; i < steps; ++i) {
        // np.linspace(0, steps, steps)[i] = i * steps/(steps-1)
        double x = (double)i * ((double)steps / (double)(steps - 1));
        if (i == steps - 1) x = (double)steps;
        double c = cos(((x / steps) + s) / (1 + s) * M_PI * 0.5);
        acp[i] = c * c;
    }
    double a0 = acp[0];
    for (int i = 0; i < steps; ++i) acp[i] /= a0;
    std::vector<float> betas(T), alphas(T), cum(T), cumprev(T);
    for (int i = 0; i < T; ++i) {
        double b = 1.0 - acp[i + 1] / acp[i];
        if (b < 0) b = 0; if (b > 0.999) b = 0.999;
        betas[i] = (float)b;
        alphas[i] = 1.0f - betas[i];
    }
    float acc = 1.0f;
    for (int i = 0; i < T; ++i) { acc = acc * alphas[i]; cum[i] = acc; cumprev[i] = i ? cum[i - 1] : 1.0f; }
    for (int i = 0; i < T; ++i) {
        float one_m = 1.0f - cum[i];
        out[SCH_BETAS * T + i] = betas[i];
        out[SCH_ACP * T + i] = cum[i];
        out[SCH_SQRT_ACP * T + i] = sqrtf(cum[i]);
        out[SCH_SQRT_1M_ACP * T + i] = sqrtf(one_m);
        float recip = 1.0f / cum[i];
        out[SCH_SQRT_RECIP * T + i] = sqrtf(recip);
        out[SCH_SQRT_RECIPM1 * T + i] = sqrtf(recip - 1.0f);
        float var = (betas[i] * (1.0f - cumprev[i])) / one_m;
        out[SCH_LOGVAR * T + i] = logf(fmaxf(var, 1e-20f));
        out[SCH_COEF1 * T + i] = (betas[i] * sqrtf(cumprev[i])) / one_m;
        out[SCH_COEF2 * T + i] = ((1.0f - cumprev[i]) * sqrtf(alphas[i])) / one_m;
    }
    return 0;
}

// ------------------------------------------------------------------ geometry
static int make_geom(const dppo_cfg* c, Geom* g) {
    if (c->obs_dim < 1 || c->action_dim < 1 || c->horizon_steps < 1 || c->cond_steps < 1) return -1;
    if (c->denoising_steps < 1 || c->denoising_steps > 255 || c->ft_denoising_steps < 0 || c->ft_denoising_steps > c->denoising_steps) return -1;
    if (c->time_dim < 4 || (c->time_dim & 1) || c->time_dim > 64) return -1;
    if (c->actor_hidden < 16 || c->actor_hidden > 1024 || c->critic_hidden < 16 || c->critic_hidden > 1024) return -1;
    if ((c->actor_hidden % 4) || (c->critic_hidden % 4)) return -1;
    g->Do = c->obs_dim * c->cond_steps; g->A = c->action_dim * c->horizon_steps;
    g->T = c->denoising_steps; g->K = c->ft_denoising_steps; g->td = c->time_dim;
    g->H = c->actor_hidden; g->Hc = c->critic_hidden;
    g->Din = g->A + g->td + g->Do;
    g->KP = round_up(g->A + g->Do, 4); g->KPc = round_up(g->Do, 4);
    size_t o = 0; const size_t td = g->td, H = g->H, A = g->A, Hc = g->Hc;
    g->ao.tw1 = o; o += td * 2 * td; g->ao.tb1 = o; o += 2 * td;
    g->ao.tw2 = o; o += 2 * td * td; g->ao.tb2 = o; o += td;
    g->ao.win = o; o += (size_t)g->Din * H; g->ao.bin = o; o += H;
    g->ao.w1 = o; o += H * H; g->ao.b1 = o; o += H;
    g->ao.w2 = o; o += H * H; g->ao.b2 = o; o += H;
    g->ao.w3 = o; o += H * A; g->ao.b3 = o; o += A;
    g->ao.n = o;
    o = 0;
    g->co.win = o; o += (size_t)g->Do * Hc; g->co.bin = o; o += Hc;
    g->co.w1 = o; o += Hc * Hc; g->co.b1 = o; o += Hc;
    g->co.w2 = o; o += Hc * Hc; g->co.b2 = o; o += Hc;
    g->co.w3 = o; o += Hc; g->co.b3 = o; o += 1;
    g->co.n = o;
    return 0;
}
extern "C" size_t dppo_num_params(const dppo_cfg* cfg, int net) {
    Geom g; if (!cfg || make_geom(cfg, &g)) return 0;
    return net == DPPO_NET_CRITIC ? g.co.n : g.ao.n;
}

// ------------------------------------------------------------------ workspace
// the old buffer may still be in use by queued work: synchronise before freeing it
int ws_reserve(Workspace& w, size_t bytes, cudaStream_t s) {
    if (bytes <= w.cap) return 0;
    if (w.base) { CUDA_TRY(cudaStreamSynchronize(s)); CUDA_TRY(cudaDeviceSynchronize()); CUDA_TRY(cudaFree(w.base)); w.base = nullptr; w.cap = 0; }
    size_t cap = bytes + (bytes >> 3) + (1 << 20);
    CUDA_TRY(cudaMalloc(&w.base, cap));
    w.cap = cap;
    return 0;
}

// ------------------------------------------------------------------ live GEMM timing
static int prof_flush(dppo_handle* h) {
    for (size_t i = 0; i + 1 < h->prof_used; i += 2) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, h->prof_ev[i], h->prof_ev[i + 1]) == cudaSuccess) h->prof_ms_acc[h->prof_cls[i / 2]] += ms;
    }
    h->prof_used = 0;
    return 0;
}
void prof_begin(dppo_handle* h, cudaStream_t s) {
    if (!h->prof_on) return;
    if (h->prof_used + 2 > h->prof_ev.size()) {
        if (h->prof_ev.size() >= 8192) { cudaDeviceSynchronize(); prof_flush(h); }
        else { for (int i = 0; i < 2; ++i) { cudaEvent_t e; cudaEventCreate(&e); h->prof_ev.push_back(e); } h->prof_cls.push_back(0); }
    }
    cudaEventRecord(h->prof_ev[h->prof_used], s);
}
void prof_end(dppo_handle* h, cudaStream_t s, double flops, int cls, double exec_flops) {
    if (!h->prof_on) return;
    cudaEventRecord(h->prof_ev[h->prof_used + 1], s);
    h->prof_cls[h->prof_used / 2] = cls;
    h->prof_used += 2; h->prof_launches[cls] += 1; h->prof_flops[cls] += flops; h->prof_exec[cls] += exec_flops >= 0 ? exec_flops : flops;
}
extern "C" int dppo_profile_enable(dppo_handle* h, int on) {
    if (!h) DPPO_FAIL(-1, "null handle");
    CUDA_TRY(cudaSetDevice(h->device)); CUDA_TRY(cudaDeviceSynchronize());
    h->prof_used = 0;
    for (int c = 0; c < 4; ++c) { h->prof_flops[c] = 0; h->prof_ms_acc[c] = 0; h->prof_launches[c] = 0; h->prof_exec[c] = 0; }
    h->prof_on = on ? 1 : 0;
    return 0;
}
extern "C" int dppo_profile_read_class(dppo_handle* h, int cls, double* ms, int64_t* launches, double* flops) {
    if (!h || cls < 0 || cls > 3) DPPO_FAIL(-1, "dppo_profile_read_class: bad arguments");
    CUDA_TRY(cudaSetDevice(h->device)); CUDA_TRY(cudaDeviceSynchronize());
    prof_flush(h);
    if (ms) *ms = h->prof_ms_acc[cls]; if (launches) *launches = h->prof_launches[cls]; if (flops) *flops = h->prof_flops[cls];
    return 0;
}
extern "C" int dppo_profile_read_exec(dppo_handle* h, int cls, double* exec_flops) {
    if (!h || cls < 0 || cls > 3 || !exec_flops) DPPO_FAIL(-1, "dppo_profile_read_exec: bad arguments");
    *exec_flops = h->prof_exec[cls];
    return 0;
}
extern "C" int dppo_profile_read(dppo_handle* h, double* ms, int64_t* launches, double* flops) {
    if (!h) DPPO_FAIL(-1, "null handle");
    CUDA_TRY(cudaSetDevice(h->device)); CUDA_TRY(cudaDeviceSynchronize());
    prof_flush(h);
    if (ms) *ms = h->prof_ms_acc[0] + h->prof_ms_acc[1] + h->prof_ms_acc[2] + h->prof_ms_acc[3];
    if (launches) *launches = h->prof_launches[0] + h->prof_launches[1] + h->prof_launches[2] + h->prof_launches[3];
    if (flops) *flops = h->prof_flops[0] + h->prof_flops[1] + h->prof_flops[2] + h->prof_flops[3];
    return 0;
}

static inline bool al16(const void* p) { return (((uintptr_t)p) & 15) == 0; }

// ------------------------------------------------------------------ SGEMM dispatch
static int gemm(dppo_handle* h, cudaStream_t s, bool a_km, bool b_nk, GemmP p, int splits = 1) {
    if (p.M <= 0 || p.N <= 0) return 0;
    const int BN = p.N <= 32 ? 32 : 128;
    if (splits < 1) splits = 1;
    int kchunk = round_up((p.K + splits - 1) / splits, 16);
    if (kchunk < 16) kchunk = 16;
    splits = (p.K + kchunk - 1) / kchunk; if (splits < 1) splits = 1;
    p.kchunk = kchunk;
    if (splits == 1) p.cstride = 0;
    p.vecA = a_km ? (p.lda % 4 == 0 && p.M % 4 == 0 && al16(p.A)) : (p.lda % 4 == 0 && p.K % 4 == 0 && al16(p.A));
    p.vecB = b_nk ? (p.ldb % 4 == 0 && p.K % 4 == 0 && al16(p.B)) : (p.ldb % 4 == 0 && p.N % 4 == 0 && al16(p.B));
    p.vecC = (p.ldc % 4 == 0 && al16(p.C) && p.cstride % 4 == 0);
    dim3 grid((p.N + BN - 1) / BN, (p.M + 127) / 128, splits);
    prof_begin(h, s);
#define SG(AK, BK_, BNV) sgemm_kernel<AK, BK_, BNV><<<grid, 256, 0, s>>>(p)
    if (BN == 128) {
        if (!a_km && !b_nk) SG(false, false, 128); else if (!a_km && b_nk) SG(false, true, 128);
        else if (a_km && !b_nk) SG(true, false, 128); else SG(true, true, 128);
    } else {
        if (!a_km && !b_nk) SG(false, false, 32); else if (!a_km && b_nk) SG(false, true, 32);
        else if (a_km && !b_nk) SG(true, false, 32); else SG(true, true, 32);
    }
#undef SG
    prof_end(h, s, 2.0 * (double)p.M * (double)p.N * (double)p.K, 2);
    KLAUNCH(h); KCHECK();
    return splits;
}
static GemmP gp(const float* A, int lda, const float* B, int ldb, float* C, int ldc, int M, int N, int K) {
    GemmP p; memset(&p, 0, sizeof(p));
    p.A = A; p.lda = lda; p.B = B; p.ldb = ldb; p.C = C; p.ldc = ldc; p.M = M; p.N = N; p.K = K; p.tconst = 0;
    return p;
}
static inline int nblk(size_t n, int b) { return (int)((n + b - 1) / b); }

// ------------------------------------------------------------------ derived tables
// w0p (the packed fp32 layer-0 weight of the FFMA path) is rebuilt lazily: the tensor mode rarely needs it
static int ensure_w0p(dppo_handle* h, int net, cudaStream_t s) {
    const Geom& g = h->g;
    if (!h->w0p_dirty[net]) return 0;
    if (net == DPPO_NET_CRITIC)
        pack_w0_kernel<<<nblk((size_t)g.KPc * g.Hc, 256), 256, 0, s>>>(h->net_w[net] + g.co.win, 0, 0, g.Do, g.KPc, g.Hc, h->ad[net].w0p);
    else
        pack_w0_kernel<<<nblk((size_t)g.KP * g.H, 256), 256, 0, s>>>(h->net_w[net] + g.ao.win, g.A, g.td, g.Do, g.KP, g.H, h->ad[net].w0p);
    KLAUNCH(h); KCHECK();
    h->w0p_dirty[net] = 0;
    return 0;
}
static int prep_net(dppo_handle* h, int net, cudaStream_t s) {
    const Geom& g = h->g;
    h->w0p_dirty[net] = 1; h->w23_dirty[net] = 1;
    if (net != DPPO_NET_CRITIC) {
        ActorDerived& d = h->ad[net];
        int threads = g.H < 64 ? 64 : (g.H > 512 ? 512 : round_up(g.H, 32));
        if (threads < 2 * g.td) threads = round_up(2 * g.td, 32);
        actor_prep_kernel<<<g.T, threads, 4 * g.td * sizeof(float), s>>>(h->net_w[net], g.ao, g.A, g.td, g.H, d.sinemb, d.thpre, d.temb, d.bt);
        KLAUNCH(h); KCHECK();
    }
    if (h->cfg.precision == DPPO_PREC_FP32) DPPO_TRY(ensure_w0p(h, net, s));
    DPPO_TRY(ts_refresh_net(h, net, s));
    return tc_refresh_net(h, net, s);
}

// ------------------------------------------------------------------ create / destroy
static int dppo_create_impl(const dppo_cfg* cfg, int device, dppo_handle** out, dppo_handle** partial);
extern "C" int dppo_create(const dppo_cfg* cfg, int device, dppo_handle** out) {
    if (!cfg || !out) DPPO_FAIL(-1, "dppo_create: null argument");
    dppo_handle* partial = nullptr;
    const int r = dppo_create_impl(cfg, device, out, &partial);
    if (r != 0 && partial) { std::string msg = dppo_last_error(); dppo_destroy(partial); dppo_set_error("%s", msg.c_str()); }   // every failure path frees what was allocated
    return r;
}
static int dppo_create_impl(const dppo_cfg* cfg, int device, dppo_handle** out, dppo_handle** partial) {
    Geom g;
    if (make_geom(cfg, &g)) DPPO_FAIL(-1, "dppo_create: invalid configuration");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) DPPO_FAIL(-4, "dppo_create: no CUDA device (%s); this library has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) DPPO_FAIL(-1, "dppo_create: device %d out of range (%d devices)", device, ndev);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop; CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) DPPO_FAIL(-4, "dppo_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    dppo_handle* h = new dppo_handle();
    *partial = h;
    h->cfg = *cfg; h->device = device; h->g = g; h->sm_count = prop.multiProcessorCount;
    { const char* tv = getenv("DPPO_PEER_TIMEOUT_S"); double sec = tv ? atof(tv) : 600.0; if (!(sec > 0)) sec = 600.0;
      h->peer_timeout_cycles = (long long)(sec * 1e3 * (double)prop.clockRate); }
    { const char* dv = getenv("DPPO_DETERMINISTIC"); h->deterministic = (dv && dv[0] == '1') ? 1 : 0; }
    const size_t nA = g.ao.n, nC = g.co.n;
    const size_t total = 3 * nA + nC;
    CUDA_TRY(cudaMalloc(&h->params, total * sizeof(float)));
    CUDA_TRY(cudaMemset(h->params, 0, total * sizeof(float)));
    h->net_w[DPPO_NET_ACTOR] = h->params; h->net_n[DPPO_NET_ACTOR] = nA;
    h->net_w[DPPO_NET_ACTOR_FT] = h->params + nA; h->net_n[DPPO_NET_ACTOR_FT] = nA;
    h->net_w[DPPO_NET_CRITIC] = h->params + 2 * nA; h->net_n[DPPO_NET_CRITIC] = nC;
    h->net_w[DPPO_NET_ACTOR_EMA] = h->params + 2 * nA + nC; h->net_n[DPPO_NET_ACTOR_EMA] = nA;
    for (int net = 0; net < 4; ++net) {
        ActorDerived& d = h->ad[net];
        memset(&d, 0, sizeof(d));
        if (net == DPPO_NET_CRITIC) { CUDA_TRY(cudaMalloc(&d.w0p, (size_t)g.KPc * g.Hc * sizeof(float))); continue; }
        CUDA_TRY(cudaMalloc(&d.sinemb, (size_t)g.T * g.td * sizeof(float)));
        CUDA_TRY(cudaMalloc(&d.thpre, (size_t)g.T * 2 * g.td * sizeof(float)));
        CUDA_TRY(cudaMalloc(&d.temb, (size_t)g.T * g.td * sizeof(float)));
        CUDA_TRY(cudaMalloc(&d.bt, (size_t)g.T * g.H * sizeof(float)));
        CUDA_TRY(cudaMalloc(&d.dte, ((size_t)g.T * g.td + 4) * sizeof(float))); CUDA_TRY(cudaMemset(d.dte, 0, ((size_t)g.T * g.td + 4) * sizeof(float)));
        CUDA_TRY(cudaMalloc(&d.w23, (size_t)g.H * g.A * sizeof(float))); CUDA_TRY(cudaMalloc(&d.b23, (size_t)g.A * sizeof(float)));
        CUDA_TRY(cudaMalloc(&d.w0p, (size_t)g.KP * g.H * sizeof(float)));
    }
    DPPO_TRY(dppo_ddpm_schedule(g.T, h->sched_host));
    CUDA_TRY(cudaMalloc(&h->sched, SCH_ROWS * g.T * sizeof(float)));
    CUDA_TRY(cudaMemcpy(h->sched, h->sched_host, SCH_ROWS * g.T * sizeof(float), cudaMemcpyHostToDevice));
    size_t on[2] = {nA, nA + nC};
    for (int i = 0; i < 2; ++i) {
        h->opt[i].n = on[i]; h->opt[i].step = 0;
        CUDA_TRY(cudaMalloc(&h->opt[i].m, on[i] * sizeof(float))); CUDA_TRY(cudaMemset(h->opt[i].m, 0, on[i] * sizeof(float)));
        CUDA_TRY(cudaMalloc(&h->opt[i].v, on[i] * sizeof(float))); CUDA_TRY(cudaMemset(h->opt[i].v, 0, on[i] * sizeof(float)));
    }
    CUDA_TRY(cudaMalloc(&h->grads, (nA + nC + 16) * sizeof(float)));
    CUDA_TRY(cudaMemset(h->grads, 0, (nA + nC + 16) * sizeof(float)));
    h->grads_buf[0] = h->grads; h->grads_floats = nA + nC + 16;
    CUDA_TRY(cudaMalloc(&h->scalars, 64 * sizeof(float)));
    CUDA_TRY(cudaMemset(h->scalars, 0, 64 * sizeof(float)));
    h->comm_status = reinterpret_cast<int*>(h->scalars + 32);
    DPPO_TRY(tc_init(h));
    DPPO_TRY(ts_init(h));
    for (int net = 0; net < 4; ++net) DPPO_TRY(prep_net(h, net, 0));
    CUDA_TRY(cudaDeviceSynchronize());
    *out = h; *partial = nullptr;
    return 0;
}
extern "C" void dppo_destroy(dppo_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    tc_plan_free(h);
    tc_destroy(h);
    ts_destroy(h);
    for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
    if (h->comm) {
        void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
        if (lib) { typedef int (*fn_t)(void*); fn_t f = (fn_t)dlsym(lib, "ncclCommDestroy"); if (f) f(h->comm); }
    }
    if (h->peers_attached) {
        for (int p = 0; p < h->world; ++p) if (p != h->rank) {
            cudaIpcCloseMemHandle(h->peer_grads[0][p]); cudaIpcCloseMemHandle(h->peer_grads[1][p]); cudaIpcCloseMemHandle(h->peer_flags[p]);
        }
    }
    cudaFree(h->env_norm);
    cudaFree(h->params); cudaFree(h->sched); cudaFree(h->grads_buf[0]); cudaFree(h->grads_buf[1]); /* gsum lives inside grads_buf[1] */ cudaFree(h->flags); cudaFree(h->scalars);
    for (int i = 0; i < 2; ++i) { cudaFree(h->opt[i].m); cudaFree(h->opt[i].v); }
    for (int net = 0; net < 4; ++net) { ActorDerived& d = h->ad[net]; cudaFree(d.sinemb); cudaFree(d.thpre); cudaFree(d.temb); cudaFree(d.bt); cudaFree(d.dte); cudaFree(d.w0p); cudaFree(d.w23); cudaFree(d.b23); }
    if (h->ws.base) cudaFree(h->ws.base);
    if (h->copy_stream) { cudaStreamDestroy(h->copy_stream); for (int i = 0; i < 9; ++i) cudaEventDestroy(h->copy_ev[i]); }
    if (h->aux_stream) { cudaStreamDestroy(h->aux_stream); for (int i = 0; i < 3; ++i) if (h->aux_ev[i]) cudaEventDestroy(h->aux_ev[i]); }
    if (h->stage.base) cudaFree(h->stage.base);
    delete h;
}

#define ENTER(h) do { if (!(h)) DPPO_FAIL(-1, "null handle"); CUDA_TRY(cudaSetDevice((h)->device)); } while (0)

extern "C" int dppo_set_weights(dppo_handle* h, int net, const float* src, size_t n, int is_device, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st;
    if (net < 0 || net > 3 || !src) DPPO_FAIL(-1, "dppo_set_weights: bad net %d", net);
    if (n != h->net_n[net]) DPPO_FAIL(-1, "dppo_set_weights: net %d has %zu parameters, got %zu", net, h->net_n[net], n);
    CUDA_TRY(cudaMemcpyAsync(h->net_w[net], src, n * sizeof(float), is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
    if (!is_device) CUDA_TRY(cudaStreamSynchronize(s));
    return prep_net(h, net, s);
}
extern "C" int dppo_get_weights(dppo_handle* h, int net, float* dst, size_t n, int is_device, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st;
    if (net < 0 || net > 3 || !dst) DPPO_FAIL(-1, "dppo_get_weights: bad net %d", net);
    if (n != h->net_n[net]) DPPO_FAIL(-1, "dppo_get_weights: net %d has %zu parameters, got %zu", net, h->net_n[net], n);
    CUDA_TRY(cudaMemcpyAsync(dst, h->net_w[net], n * sizeof(float), is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
    if (!is_device) CUDA_TRY(cudaStreamSynchronize(s));
    return 0;
}
extern "C" int dppo_set_opt_state(dppo_handle* h, int opt, const float* m, const float* v, size_t n, int64_t step, int is_device, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st;
    if (opt < 0 || opt > 1 || n != h->opt[opt].n) DPPO_FAIL(-1, "dppo_set_opt_state: bad slot/size");
    cudaMemcpyKind k = is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (m) CUDA_TRY(cudaMemcpyAsync(h->opt[opt].m, m, n * sizeof(float), k, s));
    if (v) CUDA_TRY(cudaMemcpyAsync(h->opt[opt].v, v, n * sizeof(float), k, s));
    h->opt[opt].step = step;
    if (!is_device) CUDA_TRY(cudaStreamSynchronize(s));
    return 0;
}
extern "C" int dppo_get_opt_state(dppo_handle* h, int opt, float* m, float* v, size_t n, int64_t* step, int is_device, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st;
    if (opt < 0 || opt > 1 || n != h->opt[opt].n) DPPO_FAIL(-1, "dppo_get_opt_state: bad slot/size");
    cudaMemcpyKind k = is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    if (m) CUDA_TRY(cudaMemcpyAsync(m, h->opt[opt].m, n * sizeof(float), k, s));
    if (v) CUDA_TRY(cudaMemcpyAsync(v, h->opt[opt].v, n * sizeof(float), k, s));
    if (step) *step = h->opt[opt].step;
    if (!is_device) CUDA_TRY(cudaStreamSynchronize(s));
    return 0;
}
extern "C" int dppo_set_ft_denoising_steps(dppo_handle* h, int K) {
    if (!h) DPPO_FAIL(-1, "null handle");
    if (K < 0 || K > h->g.T) DPPO_FAIL(-1, "dppo_set_ft_denoising_steps: K=%d outside [0,%d]", K, h->g.T);
    h->g.K = K; h->cfg.ft_denoising_steps = K;
    return 0;
}
extern "C" int dppo_set_grad_clip_norm(dppo_handle* h, float clip_norm) {
    if (!h) DPPO_FAIL(-1, "null handle");
    if (clip_norm != clip_norm) DPPO_FAIL(-1, "dppo_set_grad_clip_norm: NaN");
    h->grad_clip_norm = clip_norm > 0.f ? clip_norm : 0.f;
    return 0;
}
extern "C" int64_t dppo_launch_count(dppo_handle* h) { return h ? h->launches : -1; }
extern "C" int64_t dppo_tc_launch_count(dppo_handle* h) { return h ? h->tc_launches : -1; }
extern "C" int64_t dppo_fused_launch_count(dppo_handle* h) { return h ? h->fused_launches : -1; }
extern "C" int dppo_last_path(dppo_handle* h) { return h ? h->last_path : -1; }

// ------------------------------------------------------------------ fp32 layer-by-layer forward
struct FwdBufs { float *h0p, *u, *h1, *v, *out; };

static void fwd_take(dppo_handle* h, int N, int KP, int H, int NO, FwdBufs& b) {
    b.h0p = ws_take<float>(h, (size_t)N * KP);
    b.u = ws_take<float>(h, (size_t)N * H); b.h1 = ws_take<float>(h, (size_t)N * H); b.v = ws_take<float>(h, (size_t)N * H);
    b.out = ws_take<float>(h, (size_t)N * NO);
}
// actor: out[N][A] = eps; x[N][A], obs row = r / obs_div; t from trow[] or tconst
static int actor_fwd_fp32(dppo_handle* h, cudaStream_t s, int net, const float* x, const float* obs, int obs_div, int N,
                          const int* trow, int tconst, FwdBufs& b) {
    const Geom& g = h->g; const float* w = h->net_w[net]; const ActorDerived& d = h->ad[net];
    const int act1 = h->cfg.actor_act + 1;
    DPPO_TRY(ensure_w0p(h, net, s));
    pack_h0_kernel<<<nblk((size_t)N * g.KP, 256), 256, 0, s>>>(x, obs, N, g.A, g.Do, g.KP, obs_div, b.h0p); KLAUNCH(h); KCHECK();
    GemmP p = gp(b.h0p, g.KP, d.w0p, g.H, b.u, g.H, N, g.H, g.KP);
    p.btab = d.bt; p.ldbt = g.H; p.trow = trow; p.tconst = tconst;
    DPPO_TRY(gemm(h, s, false, false, p) < 0 ? -3 : 0);
    p = gp(b.u, g.H, w + g.ao.w1, g.H, b.h1, g.H, N, g.H, g.H); p.aop = act1; p.bias = w + g.ao.b1;
    DPPO_TRY(gemm(h, s, false, false, p) < 0 ? -3 : 0);
    p = gp(b.h1, g.H, w + g.ao.w2, g.H, b.v, g.H, N, g.H, g.H); p.aop = act1; p.bias = w + g.ao.b2; p.add = b.u; p.ldadd = g.H;
    DPPO_TRY(gemm(h, s, false, false, p) < 0 ? -3 : 0);
    p = gp(b.v, g.H, w + g.ao.w3, g.A, b.out, g.A, N, g.A, g.H); p.bias = w + g.ao.b3;
    DPPO_TRY(gemm(h, s, false, false, p) < 0 ? -3 : 0);
    return 0;
}
static int critic_fwd_fp32(dppo_handle* h, cudaStream_t s, const float* obs, int N, FwdBufs& b) {
    const Geom& g = h->g; const float* w = h->net_w[DPPO_NET_CRITIC]; const ActorDerived& d = h->ad[DPPO_NET_CRITIC];
    const int act1 = h->cfg.critic_act + 1;
    DPPO_TRY(ensure_w0p(h, DPPO_NET_CRITIC, s));
    pack_h0_kernel<<<nblk((size_t)N * g.KPc, 256), 256, 0, s>>>(nullptr, obs, N, 0, g.Do, g.KPc, 1, b.h0p); KLAUNCH(h); KCHECK();
    GemmP p = gp(b.h0p, g.KPc, d.w0p, g.Hc, b.u, g.Hc, N, g.Hc, g.KPc); p.bias = w + g.co.bin;
    DPPO_TRY(gemm(h, s, false, false, p) < 0 ? -3 : 0);
    p = gp(b.u, g.Hc, w + g.co.w1, g.Hc, b.h1, g.Hc, N, g.Hc, g.Hc); p.aop = act1; p.bias = w + g.co.b1;
    DPPO_TRY(gemm(h, s, false, false, p) < 0 ? -3 : 0);
    p = gp(b.h1, g.Hc, w + g.co.w2, g.Hc, b.v, g.Hc, N, g.Hc, g.Hc); p.aop = act1; p.bias = w + g.co.b2; p.add = b.u; p.ldadd = g.Hc;
    DPPO_TRY(gemm(h, s, false, false, p) < 0 ? -3 : 0);
    p = gp(b.v, g.Hc, w + g.co.w3, 1, b.out, 1, N, 1, g.Hc); p.bias = w + g.co.b3;
    DPPO_TRY(gemm(h, s, false, false, p) < 0 ? -3 : 0);
    return 0;
}

// ------------------------------------------------------------------ fp32 backward (shared by actor / critic)
struct BwdBufs { float *dv, *dh1, *du, *part; size_t part_floats; };
static int colsum(dppo_handle* h, cudaStream_t s, const float* D, int ld, int N, int ncols, const int* seg, int nseg,
                  float* part, float* out) {
    int nb = (N + 127) / 128; if (nb > 320) nb = 320; if (nb < 1) nb = 1;
    int rpb = (N + nb - 1) / nb; nb = (N + rpb - 1) / rpb;
    size_t sm = (size_t)nseg * ncols * sizeof(float);
    if (sm > 48 * 1024) {
        if (sm > 200 * 1024) DPPO_FAIL(-1, "colsum: %d segments x %d columns does not fit in shared memory", nseg, ncols);
        CUDA_TRY(cudaFuncSetAttribute(colsum_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    }
    colsum_kernel<<<nb, 256, sm, s>>>(D, ld, N, ncols, seg, nseg, rpb, part); KLAUNCH(h); KCHECK();
    size_t n = (size_t)nseg * ncols;
    tc_reduce_cols_kernel<<<nblk(n, 8), 256, 0, s>>>(part, nb, n, (int)n, out); KLAUNCH(h); KCHECK();
    return 0;
}
// dW[M=in][N=out] = aop(X)[rows][in]^T @ D[rows][out], split over rows, deterministic reduce into out
static int gemm_dw(dppo_handle* h, cudaStream_t s, const float* X, int ldx, int aop, const float* D, int ldd,
                   int rows, int M, int N, float* part, float* out) {
    int tiles = ((M + 127) / 128) * ((N + (N <= 32 ? 31 : 127)) / (N <= 32 ? 32 : 128));
    int splits = (2 * h->sm_count + tiles - 1) / tiles;
    if (splits > 40) splits = 40;
    int maxs = (rows + 255) / 256; if (splits > maxs) splits = maxs; if (splits < 1) splits = 1;
    GemmP p = gp(X, ldx, D, ldd, part, N, M, N, rows); p.aop = aop; p.cstride = (size_t)M * N;
    int S = gemm(h, s, true, false, p, splits);
    if (S < 0) return -3;
    size_t n = (size_t)M * N;
    reduce_partials_kernel<<<nblk(n, 256), 256, 0, s>>>(part, S, n, n, out, 1.f); KLAUNCH(h); KCHECK();
    return 0;
}
// generic residual-MLP backward. dout [N][NO]; writes gradient of W1,b1,W2,b2,W3,b3 into gnet at the given
// offsets, dW0p into dw0p [KP][H], and per-segment column sums of du into Gseg [nseg][H].
static int mlp_bwd_fp32(dppo_handle* h, cudaStream_t s, const float* w, size_t ow1, size_t ob1, size_t ow2, size_t ob2,
                        size_t ow3, size_t ob3, int act1, const FwdBufs& f, const float* dout, int N, int KP, int H, int NO,
                        const int* seg, int nseg, BwdBufs& b, float* gnet, float* dw0p, float* Gseg) {
    // dv = dout @ W3^T
    GemmP p = gp(dout, NO, w + ow3, NO, b.dv, H, N, H, NO);
    DPPO_TRY(gemm(h, s, false, true, p) < 0 ? -3 : 0);
    // dh1 = (dv @ W2^T) * act'(h1)
    p = gp(b.dv, H, w + ow2, H, b.dh1, H, N, H, H); p.mask = f.h1; p.ldm = H; p.mask_act = act1;
    DPPO_TRY(gemm(h, s, false, true, p) < 0 ? -3 : 0);
    // du = (dh1 @ W1^T) * act'(u) + dv
    p = gp(b.dh1, H, w + ow1, H, b.du, H, N, H, H); p.mask = f.u; p.ldm = H; p.mask_act = act1; p.add = b.dv; p.ldadd = H;
    DPPO_TRY(gemm(h, s, false, true, p) < 0 ? -3 : 0);
    // weight gradients
    DPPO_TRY(gemm_dw(h, s, f.v, H, 0, dout, NO, N, H, NO, b.part, gnet + ow3));
    DPPO_TRY(gemm_dw(h, s, f.h1, H, act1, b.dv, H, N, H, H, b.part, gnet + ow2));
    DPPO_TRY(gemm_dw(h, s, f.u, H, act1, b.dh1, H, N, H, H, b.part, gnet + ow1));
    DPPO_TRY(gemm_dw(h, s, f.h0p, KP, 0, b.du, H, N, KP, H, b.part, dw0p));
    // bias gradients
    DPPO_TRY(colsum(h, s, dout, NO, N, NO, nullptr, 1, b.part, gnet + ob3));
    DPPO_TRY(colsum(h, s, b.dv, H, N, H, nullptr, 1, b.part, gnet + ob2));
    DPPO_TRY(colsum(h, s, b.dh1, H, N, H, nullptr, 1, b.part, gnet + ob1));
    DPPO_TRY(colsum(h, s, b.du, H, N, H, seg, nseg, b.part, Gseg));
    return 0;
}
static void bwd_take(dppo_handle* h, int N, int KP, int H, int nseg, BwdBufs& b, float** Gseg, float** dw0p) {
    b.dv = ws_take<float>(h, (size_t)N * H); b.dh1 = ws_take<float>(h, (size_t)N * H); b.du = ws_take<float>(h, (size_t)N * H);
    size_t colpart = (size_t)320 * (size_t)nseg * H, gemm_part = (size_t)40 * (size_t)H * H;   // colsum / split-K partials
    b.part_floats = colpart > gemm_part ? colpart : gemm_part;
    b.part = ws_take<float>(h, b.part_floats);
    *Gseg = ws_take<float>(h, (size_t)nseg * H);
    *dw0p = ws_take<float>(h, (size_t)KP * H);
}
static int actor_bwd_fp32(dppo_handle* h, cudaStream_t s, int net, const FwdBufs& f, const float* deps, int N, const int* trow,
                          BwdBufs& b, float* Gseg, float* dw0p, float* gnet) {
    const Geom& g = h->g; const float* w = h->net_w[net];
    DPPO_TRY(mlp_bwd_fp32(h, s, w, g.ao.w1, g.ao.b1, g.ao.w2, g.ao.b2, g.ao.w3, g.ao.b3, h->cfg.actor_act + 1, f, deps, N,
                          g.KP, g.H, g.A, trow, g.T, b, gnet, dw0p, Gseg));
    CUDA_TRY(launch_time_backward(h, s, net, Gseg, gnet)); KLAUNCH(h);
    unpack_dw0_kernel<<<nblk((size_t)(g.A + g.Do) * g.H, 256), 256, 0, s>>>(dw0p, g.A, g.td, g.Do, g.H, gnet + g.ao.win); KLAUNCH(h); KCHECK();
    return 0;
}
static int critic_bwd_fp32(dppo_handle* h, cudaStream_t s, const FwdBufs& f, const float* dval, int N,
                           BwdBufs& b, float* Gseg, float* dw0p, float* gnet) {
    const Geom& g = h->g; const float* w = h->net_w[DPPO_NET_CRITIC];
    DPPO_TRY(mlp_bwd_fp32(h, s, w, g.co.w1, g.co.b1, g.co.w2, g.co.b2, g.co.w3, g.co.b3, h->cfg.critic_act + 1, f, dval, N,
                          g.KPc, g.Hc, 1, nullptr, 1, b, gnet, dw0p, Gseg));
    CUDA_TRY(cudaMemcpyAsync(gnet + g.co.bin, Gseg, g.Hc * sizeof(float), cudaMemcpyDeviceToDevice, s));
    unpack_dw0_kernel<<<nblk((size_t)g.Do * g.Hc, 256), 256, 0, s>>>(dw0p, 0, 0, g.Do, g.Hc, gnet + g.co.win); KLAUNCH(h); KCHECK();
    return 0;
}

// ------------------------------------------------------------------ forward-only entry points
static const int ROW_CHUNK = 1 << 18;

// room for the N-row actor forward of a tensor mode, which appends its buffers at call time (ts_actor_forward when split, else tc_actor_forward)
static void tensor_forward_room(dppo_handle* h, bool split, int N) {
    ws_room(h->ws, [&] {
        if (split) { TsMlp m; ts_actor_forward_take(h, DPPO_NET_ACTOR, N, m); }
        else { TcMlp m; tc_actor_forward_take(h, DPPO_NET_ACTOR, N, m); }
    });
}

extern "C" int dppo_actor_forward(dppo_handle* h, int net, const float* x, const int32_t* t, const float* obs,
                                  int N, float* eps, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st; const Geom& g = h->g;
    if (net < 0 || net > 3 || net == DPPO_NET_CRITIC || !x || !t || !obs || !eps || N < 0) DPPO_FAIL(-1, "dppo_actor_forward: bad arguments");
    for (int r0 = 0; r0 < N; r0 += ROW_CHUNK) {
        int n = N - r0 < ROW_CHUNK ? N - r0 : ROW_CHUNK;
        const bool split = ts_eligible(h, n);
        if (tc_eligible(h, n) || split) {
            DPPO_TRY(ws_layout(h->ws, s, [&] { tensor_forward_room(h, split, n); }));
            if (split) DPPO_TRY(ts_actor_forward(h, s, net, x + (size_t)r0 * g.A, obs + (size_t)r0 * g.Do, 1, n, t + r0, 0, eps + (size_t)r0 * g.A));
            else DPPO_TRY(tc_actor_forward(h, s, net, x + (size_t)r0 * g.A, obs + (size_t)r0 * g.Do, 1, n, t + r0, 0, eps + (size_t)r0 * g.A));
            continue;
        }
        FwdBufs b;
        DPPO_TRY(ws_layout(h->ws, s, [&] { fwd_take(h, n, g.KP, g.H, g.A, b); }));
        DPPO_TRY(actor_fwd_fp32(h, s, net, x + (size_t)r0 * g.A, obs + (size_t)r0 * g.Do, 1, n, t + r0, 0, b));
        CUDA_TRY(cudaMemcpyAsync(eps + (size_t)r0 * g.A, b.out, (size_t)n * g.A * sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
    return 0;
}
extern "C" int dppo_value(dppo_handle* h, const float* obs, int N, float* v, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st; const Geom& g = h->g;
    if (!obs || !v || N < 0) DPPO_FAIL(-1, "dppo_value: bad arguments");
    for (int r0 = 0; r0 < N; r0 += ROW_CHUNK) {
        int n = N - r0 < ROW_CHUNK ? N - r0 : ROW_CHUNK;
        if (tc_eligible(h, n)) { DPPO_TRY(tc_value(h, s, obs + (size_t)r0 * g.Do, n, v + r0)); continue; }
        if (ts_eligible(h, n)) { DPPO_TRY(ts_value(h, s, obs + (size_t)r0 * g.Do, n, v + r0)); continue; }
        FwdBufs b;
        DPPO_TRY(ws_layout(h->ws, s, [&] { fwd_take(h, n, g.KPc, g.Hc, 1, b); }));
        DPPO_TRY(critic_fwd_fp32(h, s, obs + (size_t)r0 * g.Do, n, b));
        CUDA_TRY(cudaMemcpyAsync(v + r0, b.out, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
    return 0;
}

static int logprobs_impl(dppo_handle* h, cudaStream_t s, const float* obs, const float* prev, const float* nxt,
                         const float* chains, const int* inds, int N, int use_base, float* logp) {
    const Geom& g = h->g;
    if (g.K < 1) DPPO_FAIL(-1, "log-probs need ft_denoising_steps >= 1");
    const int net = use_base ? DPPO_NET_ACTOR : DPPO_NET_ACTOR_FT;   // t < K for every row (diffusion_vpg.py:165-180)
    // chains mode processes whole chains per chunk (row = b*K + k)
    const int chunk_rows = chains ? (ROW_CHUNK / g.K) * g.K : ROW_CHUNK;
    for (int r0 = 0; r0 < N; r0 += chunk_rows) {
        int n = N - r0 < chunk_rows ? N - r0 : chunk_rows;
        const bool split = ts_eligible(h, n);
        const bool tensor = tc_eligible(h, n) || split;
        const bool fusedlp = tensor && !split && fc_ok(h);
        FwdBufs b; memset(&b, 0, sizeof(b));
        int* trow; float* pv; bf16* h0 = nullptr;
        DPPO_TRY(ws_layout(h->ws, s, [&] {
            if (tensor) b.out = ws_take<float>(h, (size_t)n * g.A); else fwd_take(h, n, g.KP, g.H, g.A, b);
            trow = ws_take<int>(h, n);
            pv = ws_take<float>(h, (size_t)n * g.A);
            if (fusedlp) h0 = ws_take<bf16>(h, (size_t)n * h->tc->KP0);
            else if (tensor) tensor_forward_room(h, split, n);
        }));
        const float* xin; const float* ob; int obs_div;
        const float* ch = nullptr;
        if (chains) {
            ch = chains + (size_t)(r0 / g.K) * (g.K + 1) * g.A;
            make_trow_kernel<<<nblk(n, 256), 256, 0, s>>>(nullptr, n, g.K, 1, trow); KLAUNCH(h); KCHECK();
            if (!fusedlp) { chains_prev_kernel<<<nblk((size_t)n * g.A, 256), 256, 0, s>>>(ch, n, g.A, g.K, pv); KLAUNCH(h); KCHECK(); }
            xin = pv; ob = obs + (size_t)(r0 / g.K) * g.Do; obs_div = g.K;
        } else {
            make_trow_kernel<<<nblk(n, 256), 256, 0, s>>>(inds + r0, n, g.K, 0, trow); KLAUNCH(h); KCHECK();
            xin = prev + (size_t)r0 * g.A; ob = obs + (size_t)r0 * g.Do; obs_div = 1;
        }
        const float* epsp;
        if (fusedlp) {
            // pack h0 straight from prev rows / the chains tensor, then forward + Gaussian log-prob in one fused launch
            tc_pack_h0_kernel<<<nblk((size_t)n * (h->tc->KP0 / 8), 256), 256, 0, s>>>(chains ? ch : prev + (size_t)r0 * g.A, ob, trow, 0, n, g.A, g.Do, g.T,
                                                                                      h->tc->KP0, obs_div, h0, chains ? g.K : 0);
            KLAUNCH(h); KCHECK();
            DPPO_TRY(fc_actor_infer(h, s, net, h0, n, fc::FINAL_LOGP, logp + (size_t)r0 * g.A, chains ? nullptr : prev + (size_t)r0 * g.A,
                                    chains ? nullptr : nxt + (size_t)r0 * g.A, ch, trow));
            continue;
        }
        if (split) { DPPO_TRY(ts_actor_forward(h, s, net, xin, ob, obs_div, n, trow, 0, b.out)); epsp = b.out; }
        else if (tensor) { DPPO_TRY(tc_actor_forward(h, s, net, xin, ob, obs_div, n, trow, 0, b.out)); epsp = b.out; }
        else { DPPO_TRY(actor_fwd_fp32(h, s, net, xin, ob, obs_div, n, trow, 0, b)); epsp = b.out; }
        logprob_kernel<<<nblk((size_t)n * g.A, 256), 256, 0, s>>>(chains ? nullptr : prev + (size_t)r0 * g.A,
            chains ? nullptr : nxt + (size_t)r0 * g.A, ch, epsp, trow, n, g.A, g.K, h->sched, g.T,
            h->cfg.denoised_clip_value, h->cfg.min_logprob_denoising_std, logp + (size_t)r0 * g.A);
        KLAUNCH(h); KCHECK();
    }
    return 0;
}
extern "C" int dppo_logprobs(dppo_handle* h, const float* obs, const float* chains, int B, int use_base_policy,
                             float* logp, dppo_stream_t st) {
    ENTER(h);
    if (!obs || !chains || !logp || B < 0) DPPO_FAIL(-1, "dppo_logprobs: bad arguments");
    if ((int64_t)B * h->g.K > 2000000000LL) DPPO_FAIL(-1, "dppo_logprobs: too many rows");
    return logprobs_impl(h, (cudaStream_t)st, obs, nullptr, nullptr, chains, nullptr, B * h->g.K, use_base_policy, logp);
}
extern "C" int dppo_logprobs_subsample(dppo_handle* h, const float* obs, const float* chains_prev, const float* chains_next,
                                       const int32_t* denoising_inds, int N, int use_base_policy, float* logp, dppo_stream_t st) {
    ENTER(h);
    if (!obs || !chains_prev || !chains_next || !denoising_inds || !logp || N < 0) DPPO_FAIL(-1, "dppo_logprobs_subsample: bad arguments");
    return logprobs_impl(h, (cudaStream_t)st, obs, chains_prev, chains_next, nullptr, denoising_inds, N, use_base_policy, logp);
}

// ------------------------------------------------------------------ sampling
// AP <= 32: every CTA computes all 512 layer-0 columns; wider chunks: each CTA its own 32, all-gathered (sample_cluster.cuh)
template <int AP, int R>
static auto cluster_kernel() {
    if constexpr (AP > 32) return sample_cluster_wide_kernel<AP, R>;
    else return sample_cluster_kernel<AP, R>;
}
template <int AP, int R>
static int launch_cluster(dppo_handle* h, cudaStream_t s, ClusterSampleP& p, int B, bool probe_only, int* max_clusters) {
    auto kern = cluster_kernel<AP, R>();
    size_t smem = (AP > 32 ? cluster_sample_wide_smem_floats<AP, R>() : cluster_sample_smem_floats<AP, R>()) * sizeof(float);
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = CS_C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1; cfg.blockDim = dim3(CS_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cfg.gridDim = dim3(CS_C * 8);
    int nc = 0;
    CUDA_TRY(cudaOccupancyMaxActiveClusters(&nc, kern, &cfg));
    if (max_clusters) *max_clusters = nc;
    if (probe_only) return 0;
    if (nc < 1) DPPO_FAIL(-5, "cluster sampler: no 16-CTA cluster can be resident");
    p.nchunks = (B + R - 1) / R;
    int ncl = p.nchunks < nc ? p.nchunks : nc;
    cfg.gridDim = dim3(CS_C * ncl);
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, (const ClusterSampleP)p));
    KLAUNCH(h);
    return 0;
}
template <int AP>
static int cluster_dispatch(dppo_handle* h, cudaStream_t s, ClusterSampleP& p, int B) {
    int nc = h->cluster_max;
    if (nc < 0) {
        DPPO_TRY((launch_cluster<AP, 8>(h, s, p, B, true, &nc)));
        h->cluster_max = nc;
    }
    if (nc < 1) DPPO_FAIL(-5, "cluster sampler unavailable on this device");
    int per = (B + nc - 1) / nc;
    if (per <= 2) return launch_cluster<AP, 2>(h, s, p, B, false, nullptr);
    if (per <= 4) return launch_cluster<AP, 4>(h, s, p, B, false, nullptr);
    if (per <= 6) return launch_cluster<AP, 6>(h, s, p, B, false, nullptr);
    return launch_cluster<AP, 8>(h, s, p, B, false, nullptr);
}

static int sample_layered_fp32(dppo_handle* h, cudaStream_t s, const float* obs, int B, int use_base, SampleHyper hp,
                               uint64_t seed, uint64_t offset, int64_t row_offset, const float* xT, const float* noise,
                               float* actions, float* chains, bool tensor) {
    const Geom& g = h->g;
    const bool split = tensor && ts_eligible(h, B);
    FwdBufs b; memset(&b, 0, sizeof(b));
    float* x;
    DPPO_TRY(ws_layout(h->ws, s, [&] {
        if (tensor) b.out = ws_take<float>(h, (size_t)B * g.A); else fwd_take(h, B, g.KP, g.H, g.A, b);
        x = ws_take<float>(h, (size_t)B * g.A);
        if (tensor) tensor_forward_room(h, split, B);
    }));
    sample_init_kernel<<<nblk((size_t)B * g.A, 256), 256, 0, s>>>(x, xT, B, g.A, seed, offset, row_offset, chains, g.K, g.K == g.T);
    KLAUNCH(h); KCHECK();
    for (int i = 0; i < g.T; ++i) {
        const int t = g.T - 1 - i;
        const int net = (t < g.K && !use_base) ? DPPO_NET_ACTOR_FT : DPPO_NET_ACTOR;
        if (split) DPPO_TRY(ts_actor_forward(h, s, net, x, obs, 1, B, nullptr, t, b.out));
        else if (tensor) DPPO_TRY(tc_actor_forward(h, s, net, x, obs, 1, B, nullptr, t, b.out));
        else DPPO_TRY(actor_fwd_fp32(h, s, net, x, obs, 1, B, nullptr, t, b));
        sample_update_kernel<<<nblk((size_t)B * g.A, 256), 256, 0, s>>>(x, b.out, noise, B, g.A, t, i, h->sched, g.T, hp,
            seed, offset, row_offset, chains, g.K, t <= g.K ? g.K - t : -1, actions);
        KLAUNCH(h); KCHECK();
    }
    return 0;
}

// ---- env-side glue (SURVEY.md 8f.4): MujocoLocomotionLowdimWrapper's normalisation around the sampler
// normalize_obs (mujoco_locomotion_lowdim.py:57-58): float64 raw observation, fp32 constants, fp32 denominator (max - min + 1e-6),
// float64 arithmetic, then the agent's cast to fp32 (train_ppo_diffusion_agent.py:111-113)
__global__ void env_normalize_obs_kernel(const double* __restrict__ raw, int n, int obs_dim, const float* __restrict__ omin, const float* __restrict__ omax,
                                         float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = i % obs_dim;
    const double den = (double)__fadd_rn(__fsub_rn(omax[j], omin[j]), 1e-6f);
    const double q = __ddiv_rn(__dsub_rn(raw[i], (double)omin[j]), den);
    out[i] = (float)__dmul_rn(2.0, __dsub_rn(q, 0.5));
}
__global__ void env_unnormalize_actions_kernel(const float* __restrict__ actions, int B, int A, int act_cols, int Da, const float* __restrict__ amin,
                                               const float* __restrict__ amax, float* __restrict__ raw) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * act_cols) return;
    const int r = i / act_cols, a = i % act_cols;
    raw[i] = env_unnormalize_action(actions[(size_t)r * A + a], amin[a % Da], amax[a % Da]);
}
struct EnvEpi { float* raw_actions; int act_steps; };
static int sample_impl(dppo_handle* h, const float* obs, int B, int deterministic, int use_base_policy,
                       float min_sampling_std, uint64_t seed, uint64_t offset, int64_t row_offset,
                       const float* xT, const float* noise, float* actions, float* chains, dppo_stream_t st, const EnvEpi* env);
extern "C" int dppo_sample(dppo_handle* h, const float* obs, int B, int deterministic, int use_base_policy,
                           float min_sampling_std, uint64_t seed, uint64_t offset, int64_t row_offset,
                           const float* xT, const float* noise, float* actions, float* chains, dppo_stream_t st) {
    return sample_impl(h, obs, B, deterministic, use_base_policy, min_sampling_std, seed, offset, row_offset, xT, noise, actions, chains, st, nullptr);
}
extern "C" int dppo_set_env_normalization(dppo_handle* h, const float* obs_min, const float* obs_max, const float* action_min, const float* action_max) {
    ENTER(h);
    if (!obs_min || !obs_max || !action_min || !action_max) DPPO_FAIL(-1, "dppo_set_env_normalization: null argument");
    const int od = h->cfg.obs_dim, ad = h->cfg.action_dim;
    if (!h->env_norm) CUDA_TRY(cudaMalloc(&h->env_norm, (size_t)(2 * od + 2 * ad) * sizeof(float)));
    CUDA_TRY(cudaMemcpy(h->env_norm, obs_min, od * sizeof(float), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(h->env_norm + od, obs_max, od * sizeof(float), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(h->env_norm + 2 * od, action_min, ad * sizeof(float), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(h->env_norm + 2 * od + ad, action_max, ad * sizeof(float), cudaMemcpyHostToDevice));
    return 0;
}
extern "C" int dppo_rollout_step(dppo_handle* h, const double* raw_obs, int E, int deterministic, int use_base_policy, float min_sampling_std,
                                 uint64_t seed, uint64_t offset, int64_t row_offset, const float* xT, const float* noise,
                                 float* obs_out, float* actions, float* chains, float* raw_actions, int act_steps, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st; const Geom& g = h->g;
    if (!raw_obs || !obs_out || !actions || !raw_actions || E < 1 || act_steps < 1 || act_steps > h->cfg.horizon_steps)
        DPPO_FAIL(-1, "dppo_rollout_step: bad arguments");
    if (!h->env_norm) DPPO_FAIL(-1, "dppo_rollout_step: call dppo_set_env_normalization first");
    const int od = h->cfg.obs_dim;
    env_normalize_obs_kernel<<<nblk((size_t)E * g.Do, 128), 128, 0, s>>>(raw_obs, E * g.Do, od, h->env_norm, h->env_norm + od, obs_out); KLAUNCH(h); KCHECK();
    EnvEpi env{raw_actions, act_steps};
    return sample_impl(h, obs_out, E, deterministic, use_base_policy, min_sampling_std, seed, offset, row_offset, xT, noise, actions, chains, st, &env);
}
static int sample_impl(dppo_handle* h, const float* obs, int B, int deterministic, int use_base_policy,
                       float min_sampling_std, uint64_t seed, uint64_t offset, int64_t row_offset,
                       const float* xT, const float* noise, float* actions, float* chains, dppo_stream_t st, const EnvEpi* env) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st; const Geom& g = h->g;
    if (!obs || !actions || B < 0) DPPO_FAIL(-1, "dppo_sample: bad arguments");
    if (B == 0) return 0;
    const int od_ = h->cfg.obs_dim, ad_ = h->cfg.action_dim;
    const float* amin = h->env_norm ? h->env_norm + 2 * od_ : nullptr; const float* amax = h->env_norm ? h->env_norm + 2 * od_ + ad_ : nullptr;
    // paths without the fused epilogue: one more small kernel after the chain
    auto env_tail = [&]() -> int {
        if (!env) return 0;
        const int ac = env->act_steps * ad_;
        env_unnormalize_actions_kernel<<<nblk((size_t)B * ac, 128), 128, 0, s>>>(actions, B, g.A, ac, ad_, amin, amax, env->raw_actions); KLAUNCH(h); KCHECK();
        return 0;
    };
    SampleHyper hp;
    hp.dcv = h->cfg.denoised_clip_value; hp.rcv = h->cfg.randn_clip_value; hp.facv = h->cfg.final_action_clip_value;
    hp.min_std = min_sampling_std >= 0.f ? min_sampling_std : h->cfg.min_sampling_denoising_std;
    hp.deterministic = deterministic;
    const bool split = ts_eligible(h, B);
    const bool tensor = tc_eligible(h, B) || split;
    const bool cluster_shape = (g.H == CS_H && g.A <= 128 && h->cfg.actor_act == DPPO_ACT_RELU && h->force_path != 2);
    // the persistent cluster kernel wins while the chain is latency bound; beyond that rows are
    // plentiful enough for real GEMM tiles.  Wide chunks cross over earlier (measured, DESIGN.md §5.3)
    const int cluster_limit = h->cfg.precision == DPPO_PREC_BF16 ? 1024 : g.A <= 32 ? 4096 : g.A <= 64 ? 2048 : 1024;
    if (cluster_shape && !tensor && (B <= cluster_limit || h->force_path == 1) && h->cluster_max != 0) {
        ClusterSampleP p; memset(&p, 0, sizeof(p));
        p.w[0] = h->net_w[DPPO_NET_ACTOR]; p.w[1] = h->net_w[DPPO_NET_ACTOR_FT];
        p.bt[0] = h->ad[DPPO_NET_ACTOR].bt; p.bt[1] = h->ad[DPPO_NET_ACTOR_FT].bt;
        DPPO_TRY(ensure_w23(h, DPPO_NET_ACTOR, s)); DPPO_TRY(ensure_w23(h, DPPO_NET_ACTOR_FT, s));
        p.w23[0] = h->ad[DPPO_NET_ACTOR].w23; p.w23[1] = h->ad[DPPO_NET_ACTOR_FT].w23;
        p.b23[0] = h->ad[DPPO_NET_ACTOR].b23; p.b23[1] = h->ad[DPPO_NET_ACTOR_FT].b23;
        p.o = g.ao; p.obs = obs; p.xT = xT; p.noise = noise; p.actions = actions; p.chains = chains; p.sch = h->sched;
        p.B = B; p.A = g.A; p.Do = g.Do; p.T = g.T; p.K = g.K; p.td = g.td; p.use_base_policy = use_base_policy;
        p.hp = hp; p.seed = seed; p.offset = offset; p.row_offset = row_offset;
        if (env) { p.raw_actions = env->raw_actions; p.act_min = amin; p.act_max = amax; p.act_cols = env->act_steps * ad_; p.Da = ad_; }
        int r = g.A <= 12 ? cluster_dispatch<12>(h, s, p, B) : g.A <= 24 ? cluster_dispatch<24>(h, s, p, B)
              : g.A <= 32 ? cluster_dispatch<32>(h, s, p, B) : g.A <= 64 ? cluster_dispatch<64>(h, s, p, B) : cluster_dispatch<128>(h, s, p, B);
        if (r == 0) { h->last_path = 1; return 0; }
        if (h->force_path == 1) return r;
        h->cluster_max = 0;   // not launchable here: remember and fall through to the layered path
        (void)cudaGetLastError();
    }
    if (tensor && !split && fc_ok(h)) {
        h->last_path = 4;
        DPPO_TRY(fc_sample(h, s, obs, B, use_base_policy, hp, seed, offset, row_offset, xT, noise, actions, chains));
        return env_tail();
    }
    h->last_path = tensor ? 3 : 2;
    DPPO_TRY(sample_layered_fp32(h, s, obs, B, use_base_policy, hp, seed, offset, row_offset, xT, noise, actions, chains, tensor));
    return env_tail();
}

extern "C" int dppo_sample_host(dppo_handle* h, const float* obs, int B, int deterministic, int use_base_policy,
                                float min_sampling_std, uint64_t seed, uint64_t offset, int64_t row_offset,
                                const float* xT, const float* noise, float* actions, float* chains, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st; const Geom& g = h->g;
    if (!obs || !actions || B < 0) DPPO_FAIL(-1, "dppo_sample_host: bad arguments");
    if (B == 0) return 0;
    float *d_obs, *d_xT, *d_act, *d_nz, *d_ch;
    DPPO_TRY(ws_layout(h->stage, s, [&] {
        Workspace& w = h->stage;
        d_obs = ws_take<float>(w, (size_t)B * g.Do);
        d_xT = ws_take<float>(w, (size_t)B * g.A); d_act = ws_take<float>(w, (size_t)B * g.A);
        d_nz = ws_take<float>(w, (size_t)g.T * B * g.A);
        d_ch = ws_take<float>(w, (size_t)B * (g.K + 1) * g.A);
    }));
    CUDA_TRY(cudaMemcpyAsync(d_obs, obs, (size_t)B * g.Do * 4, cudaMemcpyHostToDevice, s));
    if (xT) CUDA_TRY(cudaMemcpyAsync(d_xT, xT, (size_t)B * g.A * 4, cudaMemcpyHostToDevice, s));
    if (noise) CUDA_TRY(cudaMemcpyAsync(d_nz, noise, (size_t)g.T * B * g.A * 4, cudaMemcpyHostToDevice, s));
    DPPO_TRY(dppo_sample(h, d_obs, B, deterministic, use_base_policy, min_sampling_std, seed, offset, row_offset,
                         xT ? d_xT : nullptr, noise ? d_nz : nullptr, d_act, chains ? d_ch : nullptr, st));
    CUDA_TRY(cudaMemcpyAsync(actions, d_act, (size_t)B * g.A * 4, cudaMemcpyDeviceToHost, s));
    if (chains) CUDA_TRY(cudaMemcpyAsync(chains, d_ch, (size_t)B * (g.K + 1) * g.A * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return 0;
}

// ------------------------------------------------------------------ NCCL (dlopen)
struct NcclUid { char internal[128]; };
typedef int (*nccl_get_uid_t)(NcclUid*);
typedef int (*nccl_init_rank_t)(void**, int, NcclUid, int);
typedef int (*nccl_allreduce_t)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef const char* (*nccl_errstr_t)(int);
static void* g_nccl = nullptr;
static nccl_allreduce_t g_allreduce = nullptr;
static int nccl_load() {
    if (g_nccl) return 0;
    g_nccl = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!g_nccl) DPPO_FAIL(-6, "dlopen(libnccl.so.2) failed: %s", dlerror());
    g_allreduce = (nccl_allreduce_t)dlsym(g_nccl, "ncclAllReduce");
    if (!g_allreduce) DPPO_FAIL(-6, "ncclAllReduce not found in libnccl.so.2");
    return 0;
}
extern "C" int dppo_comm_unique_id(char* id128) {
    if (!id128) DPPO_FAIL(-1, "dppo_comm_unique_id: null");
    DPPO_TRY(nccl_load());
    nccl_get_uid_t f = (nccl_get_uid_t)dlsym(g_nccl, "ncclGetUniqueId");
    if (!f) DPPO_FAIL(-6, "ncclGetUniqueId not found");
    NcclUid u; int r = f(&u);
    if (r) DPPO_FAIL(-6, "ncclGetUniqueId failed (%d)", r);
    memcpy(id128, u.internal, 128);
    return 0;
}
extern "C" int dppo_comm_init(dppo_handle* h, const char* id128, int rank, int world) {
    ENTER(h);
    if (!id128 || world < 1 || rank < 0 || rank >= world) DPPO_FAIL(-1, "dppo_comm_init: bad arguments");
    if (world == 1) { h->rank = 0; h->world = 1; return 0; }
    DPPO_TRY(nccl_load());
    nccl_init_rank_t f = (nccl_init_rank_t)dlsym(g_nccl, "ncclCommInitRank");
    if (!f) DPPO_FAIL(-6, "ncclCommInitRank not found");
    NcclUid u; memcpy(u.internal, id128, 128);
    void* comm = nullptr;
    int r = f(&comm, world, u, rank);
    if (r) {
        nccl_errstr_t es = (nccl_errstr_t)dlsym(g_nccl, "ncclGetErrorString");
        DPPO_FAIL(-6, "ncclCommInitRank failed: %s", es ? es(r) : "?");
    }
    h->comm = comm; h->rank = rank; h->world = world;
    return 0;
}
extern "C" int dppo_comm_ipc_export(dppo_handle* h, char* out) {
    ENTER(h);
    if (!out) DPPO_FAIL(-1, "dppo_comm_ipc_export: null");
    if (!h->grads_buf[1]) {
        // one allocation [second gradient buffer | sum buffer]: the peers reach the sum buffer through the same IPC handle
        const size_t gf4 = (h->grads_floats + 3) & ~(size_t)3;
        CUDA_TRY(cudaMalloc(&h->grads_buf[1], 2 * gf4 * sizeof(float))); CUDA_TRY(cudaMemset(h->grads_buf[1], 0, 2 * gf4 * sizeof(float)));
        h->gsum = h->grads_buf[1] + gf4;
        CUDA_TRY(cudaMalloc(&h->flags, 8 * sizeof(unsigned long long))); CUDA_TRY(cudaMemset(h->flags, 0, 8 * sizeof(unsigned long long)));
        CUDA_TRY(cudaDeviceSynchronize());
    }
    cudaIpcMemHandle_t hd[3];
    CUDA_TRY(cudaIpcGetMemHandle(&hd[0], h->grads_buf[0]));
    CUDA_TRY(cudaIpcGetMemHandle(&hd[1], h->grads_buf[1]));
    CUDA_TRY(cudaIpcGetMemHandle(&hd[2], h->flags));
    static_assert(sizeof(cudaIpcMemHandle_t) * 3 == DPPO_IPC_BYTES, "IPC blob size");
    memcpy(out, hd, sizeof(hd));
    return 0;
}
extern "C" int dppo_comm_ipc_attach(dppo_handle* h, const char* all_blobs, int rank, int world) {
    ENTER(h);
    if (!all_blobs || world < 2 || world > 8 || rank < 0 || rank >= world) DPPO_FAIL(-1, "dppo_comm_ipc_attach: bad arguments (world must be 2..8)");
    if (!h->grads_buf[1]) DPPO_FAIL(-1, "dppo_comm_ipc_attach: call dppo_comm_ipc_export first");
    for (int p = 0; p < world; ++p) {
        const size_t gf4 = (h->grads_floats + 3) & ~(size_t)3;
        if (p == rank) { h->peer_grads[0][p] = h->grads_buf[0]; h->peer_grads[1][p] = h->grads_buf[1]; h->peer_gsum[p] = h->gsum; h->peer_flags[p] = h->flags; continue; }
        cudaIpcMemHandle_t hd[3]; memcpy(hd, all_blobs + (size_t)p * DPPO_IPC_BYTES, sizeof(hd));
        void* ptr[3];
        for (int k = 0; k < 3; ++k) {
            cudaError_t e = cudaIpcOpenMemHandle(&ptr[k], hd[k], cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) DPPO_FAIL(-6, "cudaIpcOpenMemHandle(rank %d, buffer %d) failed: %s", p, k, cudaGetErrorString(e));
        }
        h->peer_grads[0][p] = (float*)ptr[0]; h->peer_grads[1][p] = (float*)ptr[1]; h->peer_flags[p] = (unsigned long long*)ptr[2];
        h->peer_gsum[p] = (float*)ptr[1] + gf4;
    }
    h->rank = rank; h->world = world; h->peers_attached = 1;
    if (h->peer_two_shot < 0) { const char* tv = getenv("DPPO_PEER_TWO_SHOT"); h->peer_two_shot = tv ? (tv[0] == '1') : (world >= 4); }
    return 0;
}
// fused peer-memory all-reduce + AdamW: flag barrier, then every rank sums all ranks' gradient buffers (same order everywhere)
// and updates its replica.  The sum lands in h->gsum; the gradient buffers alternate so that peers can keep reading this one.
static int peer_allreduce_adamw(dppo_handle* h, cudaStream_t s, int opt, float* w, size_t n_param, size_t n_total, float lr, float wd) {
    OptState& o = h->opt[opt];
    o.step += 1;
    const float b1 = h->cfg.adam_beta1, b2 = h->cfg.adam_beta2;
    const float b1p = powf(b1, (float)o.step), b2p = powf(b2, (float)o.step);
    const float alpha = lr * sqrtf(1.f - b2p) / (1.f - b1p);
    PeerPtrs pp; memset(&pp, 0, sizeof(pp));
    for (int p = 0; p < h->world; ++p) { pp.g[p] = h->peer_grads[h->grads_cur][p]; pp.flags[p] = h->peer_flags[p]; }
    h->epoch += 1;
    peer_barrier_kernel<<<1, 32, 0, s>>>(pp, h->flags, h->rank, h->world, h->epoch, h->peer_timeout_cycles, h->comm_status); KLAUNCH(h); KCHECK();
    if (h->peer_two_shot == 1) {
        // reduce-scatter + broadcast of the sum over peer memory, second barrier, AdamW on the local copy of the sum
        PeerSums ps; memset(&ps, 0, sizeof(ps));
        for (int p = 0; p < h->world; ++p) ps.s[p] = h->peer_gsum[p];
        const size_t n4 = (n_total + 3) / 4, per = (n4 + h->world - 1) / h->world;
        int grid = (int)((per + 255) / 256); if (grid > 2 * h->sm_count) grid = 2 * h->sm_count; if (grid < 1) grid = 1;
        peer_reduce_scatter_bcast_kernel<<<grid, 256, 0, s>>>(pp, ps, h->rank, h->world, n4, h->comm_status); KLAUNCH(h); KCHECK();
        h->epoch += 1;
        peer_barrier_kernel<<<1, 32, 0, s>>>(pp, h->flags, h->rank, h->world, h->epoch, h->peer_timeout_cycles, h->comm_status); KLAUNCH(h); KCHECK();
        adamw_kernel<<<nblk(n_param, 256), 256, 0, s>>>(w, h->gsum, o.m, o.v, n_param, lr, alpha, b1, b2, h->cfg.adam_eps, wd, h->skip_update, h->comm_status); KLAUNCH(h); KCHECK();
    } else {
        peer_allreduce_adamw_kernel<<<2 * h->sm_count, 256, 0, s>>>(pp, h->world, h->gsum, w, o.m, o.v, n_param, n_total, lr, alpha, b1, b2, h->cfg.adam_eps, wd,
                                                                  h->skip_update, h->comm_status);
        KLAUNCH(h); KCHECK();
    }
    h->grads_cur ^= 1; h->grads = h->grads_buf[h->grads_cur];        // the next step accumulates into the other buffer
    return 0;
}
static int allreduce_sum(dppo_handle* h, float* buf, size_t n, cudaStream_t s) {
    if (h->world <= 1) return 0;
    if (!h->comm || !g_allreduce) DPPO_FAIL(-6, "all-reduce requested but no communicator attached");
    int r = g_allreduce(buf, buf, n, 7 /*ncclFloat32*/, 0 /*ncclSum*/, h->comm, s);
    if (r) DPPO_FAIL(-6, "ncclAllReduce failed (%d)", r);
    return 0;
}

// 0 = healthy; 1 = a peer barrier timed out (a rank died or fell more than DPPO_PEER_TIMEOUT_S behind): the updates since were skipped
extern "C" int dppo_comm_status(dppo_handle* h) {
    ENTER(h);
    int st = 0;
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(&st, h->comm_status, sizeof(int), cudaMemcpyDeviceToHost));
    if (st) DPPO_FAIL(-6, "peer-memory gradient exchange: a flag barrier timed out; weights and optimizer state were left untouched since");
    return 0;
}

// ------------------------------------------------------------------ AdamW
// advances optimizer `opt` by one step and returns that step's bias-corrected step size
static float adam_next_alpha(dppo_handle* h, int opt, float lr) {
    OptState& o = h->opt[opt];
    o.step += 1;
    const float b1p = powf(h->cfg.adam_beta1, (float)o.step), b2p = powf(h->cfg.adam_beta2, (float)o.step);
    return lr * sqrtf(1.f - b2p) / (1.f - b1p);
}
static int adam_apply(dppo_handle* h, cudaStream_t s, int opt, float* w, const float* g, size_t n, float lr, float wd) {
    OptState& o = h->opt[opt];
    const float b1 = h->cfg.adam_beta1, b2 = h->cfg.adam_beta2;
    const float alpha = adam_next_alpha(h, opt, lr);
    adamw_kernel<<<nblk(n, 256), 256, 0, s>>>(w, g, o.m, o.v, n, lr, alpha, b1, b2, h->cfg.adam_eps, wd, h->skip_update, nullptr); KLAUNCH(h); KCHECK();
    return 0;
}

// ------------------------------------------------------------------ PPO step
static int prep_net(dppo_handle* h, int net, cudaStream_t s);
// all-reduce (if a communicator is attached) + AdamW + derived-table refresh + metric / gradient read-out
// The split-precision mode applies AdamW and rebuilds every derived table in ONE launch (ts_apply_update) after a local or NCCL
// reduction; with gradient clipping or the peer-memory exchange (whose kernel fuses the reduction with AdamW) it keeps the separate
// AdamW launch and prep_net, like the other modes.
static int ppo_apply_tail(dppo_handle* h, cudaStream_t s, float lr, int apply, float* metrics8, float* grads_out) {
    const size_t nA = h->g.ao.n, nC = h->g.co.n; float* gr = h->grads;
    if (apply) {
        bool tables_done = false;
        // actor_ft and critic are contiguous in `params` and share one optimizer (train_ppo_diffusion_agent.py:354-356)
        if (h->grad_clip_norm > 0.f) {
            // clipping needs the norms of the REDUCED gradient before the update: reduce, (hand out the unclipped gradient), clip, update
            DPPO_TRY(allreduce_sum(h, gr, nA + nC + 8, s));
            if (grads_out) { CUDA_TRY(cudaMemcpyAsync(grads_out, gr, (nA + nC) * sizeof(float), cudaMemcpyDeviceToDevice, s)); grads_out = nullptr; }
            const ActorOff& a = h->g.ao; const CriticOff& c = h->g.co;
            const size_t offs[21] = {a.tw1, a.tb1, a.tw2, a.tb2, a.win, a.bin, a.w1, a.b1, a.w2, a.b2, a.w3, a.b3,
                                     nA + c.win, nA + c.bin, nA + c.w1, nA + c.b1, nA + c.w2, nA + c.b2, nA + c.w3, nA + c.b3, nA + nC};
            VarSegs segs; segs.n = 20;
            for (int i = 0; i <= 20; ++i) segs.off[i] = (unsigned int)offs[i];
            clip_by_norm_kernel<<<segs.n, 1024, 0, s>>>(gr, segs, h->grad_clip_norm); KLAUNCH(h); KCHECK();
            DPPO_TRY(adam_apply(h, s, DPPO_OPT_FINETUNE, h->net_w[DPPO_NET_ACTOR_FT], gr, nA + nC, lr, h->cfg.weight_decay));
        } else if (h->peers_attached && h->world > 1) {
            DPPO_TRY(peer_allreduce_adamw(h, s, DPPO_OPT_FINETUNE, h->net_w[DPPO_NET_ACTOR_FT], nA + nC, nA + nC + 8, lr, h->cfg.weight_decay));
            gr = h->gsum;
        } else {
            DPPO_TRY(allreduce_sum(h, gr, nA + nC + 8, s));
            if (ts_update_ok(h)) {
                DPPO_TRY(ts_apply_update(h, s, gr, lr, adam_next_alpha(h, DPPO_OPT_FINETUNE, lr), h->cfg.weight_decay, nullptr));
                tables_done = true;
            } else {
                DPPO_TRY(adam_apply(h, s, DPPO_OPT_FINETUNE, h->net_w[DPPO_NET_ACTOR_FT], gr, nA + nC, lr, h->cfg.weight_decay));
            }
        }
        if (tables_done) {
        } else if (h->cfg.precision == DPPO_PREC_BF16 && tc_shapes_ok(h) && 2 * h->g.td <= 256) {
            DPPO_TRY(tc_prep_pack_ft_critic(h, s));
        } else {
            DPPO_TRY(prep_net(h, DPPO_NET_ACTOR_FT, s));
            DPPO_TRY(prep_net(h, DPPO_NET_CRITIC, s));
        }
    }
    else if (h->world > 1) {
        // loss + gradients only (critic warm-up iterations, diagnostics): the metrics / gradients handed out are still the GLOBAL
        // ones, so that the KL early stop (train_ppo_diffusion_agent.py:366-368) is taken on the same value by every rank
        DPPO_TRY(allreduce_sum(h, gr, nA + nC + 8, s));
    }
    if (metrics8) CUDA_TRY(cudaMemcpyAsync(metrics8, gr + nA + nC, 8 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (grads_out) CUDA_TRY(cudaMemcpyAsync(grads_out, gr, (nA + nC) * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return 0;
}
extern "C" int dppo_ppo_step(dppo_handle* h, const float* obs, const float* prev, const float* nxt,
                             const int32_t* inds, const float* returns, const float* oldvalues,
                             const float* advantages, const float* oldlogp, int N, int64_t N_global,
                             float adv_mean, float adv_std, float lr, int apply,
                             float* metrics8, float* grads_out, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st; const Geom& g = h->g;
    if (!obs || !prev || !nxt || !inds || !returns || !oldvalues || !advantages || !oldlogp || N < 1 || N_global < N)
        DPPO_FAIL(-1, "dppo_ppo_step: bad arguments");
    if (g.K < 1) DPPO_FAIL(-1, "dppo_ppo_step: ft_denoising_steps must be >= 1");
    if (adv_std < 0.f && N_global != N) DPPO_FAIL(-1, "dppo_ppo_step: global advantage statistics are required when rows are sharded");
    const size_t nA = g.ao.n, nC = g.co.n;
    float* gr = h->grads;
    if (tc_eligible(h, N)) {
        DPPO_TRY(tc_ppo_step(h, s, obs, prev, nxt, inds, returns, oldvalues, advantages, oldlogp, N, N_global, adv_mean, adv_std));
    } else if (ts_eligible(h, N)) {
        DPPO_TRY(ts_ppo_step(h, s, obs, prev, nxt, inds, returns, oldvalues, advantages, oldlogp, N, N_global, adv_mean, adv_std));
    } else {
        const int nlb = nblk(N, 128);
        FwdBufs fa, fc; BwdBufs ba, bc; float *Ga, *Gc, *dw0a, *dw0c, *deps, *dval; int* trow; double* bsum;
        DPPO_TRY(ws_layout(h->ws, s, [&] {
            fwd_take(h, N, g.KP, g.H, g.A, fa); fwd_take(h, N, g.KPc, g.Hc, 1, fc);
            bwd_take(h, N, g.KP, g.H, g.T, ba, &Ga, &dw0a); bwd_take(h, N, g.KPc, g.Hc, 1, bc, &Gc, &dw0c);
            trow = ws_take<int>(h, N);
            deps = ws_take<float>(h, (size_t)N * g.A);
            dval = ws_take<float>(h, N);
            bsum = ws_take<double>(h, (size_t)nlb * 5);
        }));
        make_trow_kernel<<<nblk(N, 256), 256, 0, s>>>(inds, N, g.K, 0, trow); KLAUNCH(h); KCHECK();
        DPPO_TRY(launch_adv_stats(h, s, advantages, nullptr, N, adv_mean, adv_std));
        DPPO_TRY(actor_fwd_fp32(h, s, DPPO_NET_ACTOR_FT, prev, obs, 1, N, trow, 0, fa));
        DPPO_TRY(critic_fwd_fp32(h, s, obs, N, fc));
        const PpoHyper hp = ppo_hyper(h, N_global);
        ppo_loss_kernel<<<nlb, 128, 0, s>>>(prev, nxt, fa.out, inds, returns, oldvalues, advantages, oldlogp, fc.out,
                                           h->scalars, h->sched, hp, N, deps, dval, bsum); KLAUNCH(h); KCHECK();
        ppo_metrics_kernel<<<1, 256, 0, s>>>(bsum, nlb, hp.inv_nglobal, (float)((double)N / (double)N_global), gr + nA + nC); KLAUNCH(h); KCHECK();
        DPPO_TRY(actor_bwd_fp32(h, s, DPPO_NET_ACTOR_FT, fa, deps, N, trow, ba, Ga, dw0a, gr));
        DPPO_TRY(critic_bwd_fp32(h, s, fc, dval, N, bc, Gc, dw0c, gr + nA));
    }
    return ppo_apply_tail(h, s, lr, apply, metrics8, grads_out);
}

extern "C" int dppo_ppo_step_host(dppo_handle* h, const float* obs, const float* prev, const float* nxt,
                                  const int32_t* inds, const float* returns, const float* oldvalues,
                                  const float* advantages, const float* oldlogp, int N, int64_t N_global,
                                  float adv_mean, float adv_std, float lr, int apply, float* metrics8_host, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st; const Geom& g = h->g;
    if (N < 1) DPPO_FAIL(-1, "dppo_ppo_step_host: bad arguments");
    float *d_obs, *d_prev, *d_next, *d_olp, *d_ret, *d_val, *d_adv, *d_met; int* d_inds;
    DPPO_TRY(ws_layout(h->stage, s, [&] {
        Workspace& w = h->stage;
        d_obs = ws_take<float>(w, (size_t)N * g.Do);
        d_prev = ws_take<float>(w, (size_t)N * g.A); d_next = ws_take<float>(w, (size_t)N * g.A); d_olp = ws_take<float>(w, (size_t)N * g.A);
        d_inds = ws_take<int>(w, N); d_ret = ws_take<float>(w, N); d_val = ws_take<float>(w, N); d_adv = ws_take<float>(w, N);
        d_met = ws_take<float>(w, 8);
    }));
    // tensor mode: chunked pipeline - the H2D copy of chunk c+1 (copy stream) overlaps the compute of chunk c
    const int chunk_rows = (tc_eligible(h, N) && fc_ok(h) && fc_critic_ok(h) && !h->deterministic) ? tc_ppo_pipeline_chunk_rows(h, N) : 0;
    if (chunk_rows > 0) {
        if (!obs || !prev || !nxt || !inds || !returns || !oldvalues || !advantages || !oldlogp || N_global < N) DPPO_FAIL(-1, "dppo_ppo_step_host: bad arguments");
        if (adv_std < 0.f && N_global != N) DPPO_FAIL(-1, "dppo_ppo_step_host: global advantage statistics are required when rows are sharded");
        if (!h->copy_stream) {
            CUDA_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
            for (int i = 0; i < 9; ++i) CUDA_TRY(cudaEventCreateWithFlags(&h->copy_ev[i], cudaEventDisableTiming));
        }
        cudaStream_t cs = h->copy_stream;
        // staging is free: the previous *_host call synchronised `s`; the copy stream must still not overtake work queued on s
        CUDA_TRY(cudaEventRecord(h->copy_ev[8], s));
        CUDA_TRY(cudaStreamWaitEvent(cs, h->copy_ev[8], 0));
        // a short first chunk (a third of a wave-sized one) gets the GPU going while the bulk of the minibatch is still on the link
        const int lead = ((chunk_rows / 3) + 127) & ~127;
        DPPO_TRY(tc_ppo_begin(h, s, N, chunk_rows, N_global, lead));
        const int CR = tc_plan(h).chunk_rows, nchunks = tc_plan(h).nchunks;
        if (nchunks > 8) DPPO_FAIL(-7, "dppo_ppo_step_host: too many pipeline chunks");
        size_t cr0[8], cn[8];
        { size_t r = 0; for (int c = 0; c < nchunks; ++c) { size_t want = (c == 0 && tc_plan(h).lead_rows > 0) ? (size_t)tc_plan(h).lead_rows : (size_t)CR;
                                                            cr0[c] = r; cn[c] = r >= (size_t)N ? 0 : ((size_t)N - r < want ? (size_t)N - r : want); r += cn[c]; } }
        CUDA_TRY(cudaMemcpyAsync(d_adv, advantages, (size_t)N * 4, cudaMemcpyHostToDevice, cs));
        for (int c = 0; c < nchunks; ++c) {
            const size_t r0 = cr0[c]; if (cn[c] == 0) break;
            const size_t n = cn[c];
            CUDA_TRY(cudaMemcpyAsync(d_obs + r0 * g.Do, obs + r0 * g.Do, n * g.Do * 4, cudaMemcpyHostToDevice, cs));
            CUDA_TRY(cudaMemcpyAsync(d_prev + r0 * g.A, prev + r0 * g.A, n * g.A * 4, cudaMemcpyHostToDevice, cs));
            CUDA_TRY(cudaMemcpyAsync(d_next + r0 * g.A, nxt + r0 * g.A, n * g.A * 4, cudaMemcpyHostToDevice, cs));
            CUDA_TRY(cudaMemcpyAsync(d_olp + r0 * g.A, oldlogp + r0 * g.A, n * g.A * 4, cudaMemcpyHostToDevice, cs));
            CUDA_TRY(cudaMemcpyAsync(d_inds + r0, inds + r0, n * 4, cudaMemcpyHostToDevice, cs));
            CUDA_TRY(cudaMemcpyAsync(d_ret + r0, returns + r0, n * 4, cudaMemcpyHostToDevice, cs));
            CUDA_TRY(cudaMemcpyAsync(d_val + r0, oldvalues + r0, n * 4, cudaMemcpyHostToDevice, cs));
            CUDA_TRY(cudaEventRecord(h->copy_ev[c], cs));
        }
        for (int c = 0; c < nchunks; ++c) {
            const size_t r0 = cr0[c]; if (cn[c] == 0) break;
            const int n = (int)cn[c];
            CUDA_TRY(cudaStreamWaitEvent(s, h->copy_ev[c], 0));
            if (c == 0) DPPO_TRY(tc_ppo_adv_stats(h, s, d_adv, N, adv_mean, adv_std));     // the advantages were copied first
            DPPO_TRY(tc_ppo_chunk(h, s, c, d_obs + r0 * g.Do, d_prev + r0 * g.A, d_next + r0 * g.A, d_inds + r0, d_ret + r0, d_val + r0,
                                  d_adv + r0, d_olp + r0 * g.A, n));
        }
        DPPO_TRY(tc_ppo_finish(h, s));
        DPPO_TRY(ppo_apply_tail(h, s, lr, apply, d_met, nullptr));
    } else {
    CUDA_TRY(cudaMemcpyAsync(d_obs, obs, (size_t)N * g.Do * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_prev, prev, (size_t)N * g.A * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_next, nxt, (size_t)N * g.A * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_olp, oldlogp, (size_t)N * g.A * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_inds, inds, (size_t)N * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_ret, returns, (size_t)N * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_val, oldvalues, (size_t)N * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_adv, advantages, (size_t)N * 4, cudaMemcpyHostToDevice, s));
    DPPO_TRY(dppo_ppo_step(h, d_obs, d_prev, d_next, d_inds, d_ret, d_val, d_adv, d_olp, N, N_global, adv_mean, adv_std, lr, apply,
                           d_met, nullptr, st));
    }
    if (metrics8_host) CUDA_TRY(cudaMemcpyAsync(metrics8_host, d_met, 8 * sizeof(float), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return 0;
}

// ------------------------------------------------------------------ index-driven PPO step (SURVEY.md 8f.1)
static int ppo_indexed_impl(dppo_handle* h, cudaStream_t s, const float* obs_buf, const float* chains_buf, const float* oldlogp_buf,
                            const float* returns_buf, const float* values_buf, const float* adv_buf, int64_t P,
                            const int32_t* inds_dev, const int32_t* inds_host, int N, int64_t N_global, float adv_mean, float adv_std,
                            float lr, int apply, float* metrics8, float* grads_out, float* metrics8_host) {
    const Geom& g = h->g;
    if (!obs_buf || !chains_buf || !oldlogp_buf || !returns_buf || !values_buf || !adv_buf || (!inds_dev && !inds_host) || N < 1 || P < 1 || N_global < N)
        DPPO_FAIL(-1, "dppo_ppo_step_indexed: bad arguments");
    if (g.K < 1) DPPO_FAIL(-1, "dppo_ppo_step_indexed: ft_denoising_steps must be >= 1");
    if (P * g.K > 2000000000LL) DPPO_FAIL(-1, "dppo_ppo_step_indexed: rollout buffer too large for int32 flat indices");
    float *d_obs, *d_prev, *d_next, *d_olp, *d_ret, *d_val, *d_adv, *d_met; int *d_dind, *d_inds, *d_bad;
    DPPO_TRY(ws_layout(h->stage, s, [&] {
        Workspace& w = h->stage;
        d_obs = ws_take<float>(w, (size_t)N * g.Do);
        d_prev = ws_take<float>(w, (size_t)N * g.A); d_next = ws_take<float>(w, (size_t)N * g.A); d_olp = ws_take<float>(w, (size_t)N * g.A);
        d_dind = ws_take<int>(w, N); d_ret = ws_take<float>(w, N); d_val = ws_take<float>(w, N); d_adv = ws_take<float>(w, N);
        d_inds = ws_take<int>(w, N);
        d_met = ws_take<float>(w, 8); d_bad = ws_take<int>(w, 1);
    }));
    if (inds_host) { CUDA_TRY(cudaMemcpyAsync(d_inds, inds_host, (size_t)N * 4, cudaMemcpyHostToDevice, s)); inds_dev = d_inds; }
    CUDA_TRY(cudaMemsetAsync(d_bad, 0, sizeof(int), s));
    // tensor mode: no materialised minibatch - the h0 pack and loss kernels read the rollout buffers through the flat indices
    TcIdxView view; view.flat = inds_dev; view.K = g.K; view.P = (long long)P; view.chains = chains_buf; view.obs = obs_buf; view.olp = oldlogp_buf;
    view.ret = returns_buf; view.val = values_buf; view.adv = adv_buf; view.bad = d_bad;
    // an index outside [0, P*K) must not reach the optimizer: the pack / gather kernels raise d_bad, which turns AdamW (and the
    // operand refresh that follows) into a no-op on the device; the host variant then returns an error, the device variant
    // hands back NaN metrics
    struct SkipGuard { dppo_handle* h; ~SkipGuard() { h->skip_update = nullptr; } } guard{h};
    h->skip_update = d_bad;
    if (tc_eligible(h, N) && tc_ppo_indexed_ok(h, view) && (adv_std >= 0.f || N_global == N)) {
        DPPO_TRY(tc_ppo_step_indexed(h, s, view, N, N_global, adv_mean, adv_std));
        DPPO_TRY(ppo_apply_tail(h, s, lr, apply, metrics8_host ? d_met : metrics8, grads_out));
    } else if (ts_eligible(h, N) && ts_ppo_indexed_ok(h, view) && (adv_std >= 0.f || N_global == N)) {
        DPPO_TRY(ts_ppo_step(h, s, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, N, N_global, adv_mean, adv_std, &view));
        DPPO_TRY(ppo_apply_tail(h, s, lr, apply, metrics8_host ? d_met : metrics8, grads_out));
    } else {
    const size_t total = (size_t)N * (g.Do + 3 * g.A + 4);
    gather_minibatch_kernel<<<nblk(total, 256), 256, 0, s>>>(obs_buf, chains_buf, oldlogp_buf, returns_buf, values_buf, adv_buf, inds_dev, N, g.K, g.A, g.Do,
                                                           (long long)P, d_obs, d_prev, d_next, d_olp, d_dind, d_ret, d_val, d_adv, d_bad);
    KLAUNCH(h); KCHECK();
    DPPO_TRY(dppo_ppo_step(h, d_obs, d_prev, d_next, d_dind, d_ret, d_val, d_adv, d_olp, N, N_global, adv_mean, adv_std, lr, apply,
                           metrics8_host ? d_met : metrics8, grads_out, (dppo_stream_t)s));
    }
    if (!metrics8_host && metrics8) { poison_metrics_kernel<<<1, 32, 0, s>>>(metrics8, d_bad); KLAUNCH(h); KCHECK(); }
    if (metrics8_host) {
        int bad = 0;
        CUDA_TRY(cudaMemcpyAsync(metrics8_host, d_met, 8 * sizeof(float), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        if (bad) DPPO_FAIL(-1, "dppo_ppo_step_indexed_host: an index lies outside [0, P*K); the optimizer step was skipped");
    }
    return 0;
}
extern "C" int dppo_ppo_step_indexed(dppo_handle* h, const float* obs_buf, const float* chains_buf, const float* oldlogp_buf,
                                     const float* returns_buf, const float* values_buf, const float* adv_buf, int64_t P,
                                     const int32_t* inds_k, int N, int64_t N_global, float adv_mean, float adv_std, float lr, int apply,
                                     float* metrics8, float* grads_out, dppo_stream_t st) {
    ENTER(h);
    return ppo_indexed_impl(h, (cudaStream_t)st, obs_buf, chains_buf, oldlogp_buf, returns_buf, values_buf, adv_buf, P, inds_k, nullptr, N, N_global,
                            adv_mean, adv_std, lr, apply, metrics8, grads_out, nullptr);
}
extern "C" int dppo_ppo_step_indexed_host(dppo_handle* h, const float* obs_buf, const float* chains_buf, const float* oldlogp_buf,
                                          const float* returns_buf, const float* values_buf, const float* adv_buf, int64_t P,
                                          const int32_t* inds_k_host, int N, int64_t N_global, float adv_mean, float adv_std, float lr, int apply,
                                          float* metrics8_host, dppo_stream_t st) {
    ENTER(h);
    if (!metrics8_host) DPPO_FAIL(-1, "dppo_ppo_step_indexed_host: metrics8_host is required");
    return ppo_indexed_impl(h, (cudaStream_t)st, obs_buf, chains_buf, oldlogp_buf, returns_buf, values_buf, adv_buf, P, nullptr, inds_k_host, N, N_global,
                            adv_mean, adv_std, lr, apply, nullptr, nullptr, metrics8_host);
}

// ------------------------------------------------------------------ GAE (SURVEY.md 8f.2)
extern "C" int dppo_gae(dppo_handle* h, const double* rewards, const float* terminated, const float* values, const float* next_values,
                        int n_steps, int n_envs, double reward_scale_const, double gamma, double gae_lambda,
                        float* advantages, float* returns, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st;
    if (!rewards || !terminated || !values || !next_values || !advantages || !returns || n_steps < 1 || n_envs < 1)
        DPPO_FAIL(-1, "dppo_gae: bad arguments");
    gae_kernel<<<nblk(n_envs, 128), 128, 0, s>>>(rewards, terminated, values, next_values, n_steps, n_envs, reward_scale_const, gamma, gae_lambda,
                                                advantages, returns);
    KLAUNCH(h); KCHECK();
    return 0;
}

// ------------------------------------------------------------------ pre-train step
extern "C" int dppo_pretrain_step(dppo_handle* h, const float* actions, const float* obs, int N, int64_t N_global,
                                  int64_t row_offset, const int32_t* t_in, const float* noise_in,
                                  uint64_t seed, uint64_t offset, float lr, int apply,
                                  float* loss, float* grads_out, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st; const Geom& g = h->g;
    if (!actions || !obs || N < 1 || N_global < N) DPPO_FAIL(-1, "dppo_pretrain_step: bad arguments");
    const size_t nA = g.ao.n;
    float* gr = h->grads;
    if (tc_eligible(h, N)) {
        DPPO_TRY(tc_pretrain_grads(h, s, actions, obs, N, N_global, row_offset, t_in, noise_in, seed, offset));
    } else if (ts_eligible(h, N)) {
        DPPO_TRY(ts_pretrain_grads(h, s, actions, obs, N, N_global, row_offset, t_in, noise_in, seed, offset));
    } else {
        const size_t ne = (size_t)N * g.A;
        const int nlb = nblk(ne, 256);
        FwdBufs fa; BwdBufs ba; float *Ga, *dw0a, *noise, *xn, *deps; int* trow; double* bsum;
        DPPO_TRY(ws_layout(h->ws, s, [&] {
            fwd_take(h, N, g.KP, g.H, g.A, fa);
            bwd_take(h, N, g.KP, g.H, g.T, ba, &Ga, &dw0a);
            trow = ws_take<int>(h, N);
            noise = ws_take<float>(h, ne); xn = ws_take<float>(h, ne); deps = ws_take<float>(h, ne);
            bsum = ws_take<double>(h, nlb);
        }));
        pretrain_prep_kernel<<<nblk(ne, 256), 256, 0, s>>>(actions, t_in, noise_in, N, g.A, g.T, h->sched, seed, offset, row_offset, trow, noise, xn);
        KLAUNCH(h); KCHECK();
        DPPO_TRY(actor_fwd_fp32(h, s, DPPO_NET_ACTOR, xn, obs, 1, N, trow, 0, fa));
        mse_loss_kernel<<<nlb, 256, 0, s>>>(fa.out, noise, ne, 1.0f / ((float)N_global * (float)g.A), deps, bsum); KLAUNCH(h); KCHECK();
        sum_blocks_kernel<<<1, 256, 0, s>>>(bsum, nlb, 1.0f / ((float)N_global * (float)g.A), gr + nA); KLAUNCH(h); KCHECK();
        DPPO_TRY(actor_bwd_fp32(h, s, DPPO_NET_ACTOR, fa, deps, N, trow, ba, Ga, dw0a, gr));
    }
    if (apply) {
        if (h->peers_attached && h->world > 1) {
            DPPO_TRY(peer_allreduce_adamw(h, s, DPPO_OPT_PRETRAIN, h->net_w[DPPO_NET_ACTOR], nA, nA + 8, lr, h->cfg.pretrain_weight_decay));
            gr = h->gsum;
        } else {
            DPPO_TRY(allreduce_sum(h, gr, nA + 8, s));
            DPPO_TRY(adam_apply(h, s, DPPO_OPT_PRETRAIN, h->net_w[DPPO_NET_ACTOR], gr, nA, lr, h->cfg.pretrain_weight_decay));
        }
        DPPO_TRY(prep_net(h, DPPO_NET_ACTOR, s));
    }
    if (loss) CUDA_TRY(cudaMemcpyAsync(loss, gr + nA, sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (grads_out) CUDA_TRY(cudaMemcpyAsync(grads_out, gr, nA * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return 0;
}
extern "C" int dppo_ema_update(dppo_handle* h, float decay, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st;
    size_t n = h->g.ao.n;
    ema_kernel<<<nblk(n, 256), 256, 0, s>>>(h->net_w[DPPO_NET_ACTOR_EMA], h->net_w[DPPO_NET_ACTOR], n, decay); KLAUNCH(h); KCHECK();
    return prep_net(h, DPPO_NET_ACTOR_EMA, s);
}
// dev tool: enable per-CTA cycle counters of the fused chain kernel and read them back (host out [sm_count][8])
extern "C" int dppo_debug_chain_timing(dppo_handle* h, int enable, long long* out_host, int* sm_count) {
    if (!h) DPPO_FAIL(-1, "null handle");
    CUDA_TRY(cudaSetDevice(h->device));
    if (sm_count) *sm_count = h->sm_count;
    const size_t bytes = (size_t)16 * h->sm_count * 8 * sizeof(long long);     // 16 launch slots, round robin; reading resets the slot index
    if (enable && !h->chain_dbg) { CUDA_TRY(cudaMalloc(&h->chain_dbg, bytes)); CUDA_TRY(cudaMemset(h->chain_dbg, 0, bytes)); h->chain_dbg_idx = 0; }
    if (out_host && h->chain_dbg) {
        CUDA_TRY(cudaDeviceSynchronize()); CUDA_TRY(cudaMemcpy(out_host, h->chain_dbg, bytes, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemset(h->chain_dbg, 0, bytes)); h->chain_dbg_idx = 0;
    }
    if (!enable && h->chain_dbg) { CUDA_TRY(cudaDeviceSynchronize()); cudaFree(h->chain_dbg); h->chain_dbg = nullptr; }
    return 0;
}
// dev probe (tools/mma_probe.py): out_host [2*grid] per CTA, see fc::mma_probe_kernel
__global__ void __launch_bounds__(256) ffma_peak_kernel(float* __restrict__ out, int iters, float x, float y) {
    float a[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) a[j] = (float)(threadIdx.x + j) * 1e-6f;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int j = 0; j < 16; ++j) a[j] = fmaf(a[j], x, y);
    }
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 16; ++j) s += a[j];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}
extern "C" int dppo_debug_ffma_peak(dppo_handle* h, double* tflops) {
    ENTER(h);
    if (!tflops) DPPO_FAIL(-1, "dppo_debug_ffma_peak: bad arguments");
    const int blocks = h->sm_count * 8, iters = 8192;
    float* out = nullptr;
    CUDA_TRY(cudaMalloc(&out, (size_t)blocks * 256 * sizeof(float)));
    cudaEvent_t a, b; CUDA_TRY(cudaEventCreate(&a)); CUDA_TRY(cudaEventCreate(&b));
    ffma_peak_kernel<<<blocks, 256>>>(out, iters, 0.999f, 1e-3f);
    CUDA_TRY(cudaEventRecord(a, 0));
    for (int r = 0; r < 4; ++r) ffma_peak_kernel<<<blocks, 256>>>(out, iters, 0.999f, 1e-3f);
    CUDA_TRY(cudaEventRecord(b, 0));
    CUDA_TRY(cudaEventSynchronize(b));
    float ms = 0.f; CUDA_TRY(cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(out);
    *tflops = 4.0 * (double)blocks * 256.0 * (double)iters * 16.0 * 2.0 / ((double)ms * 1e-3) / 1e12;
    return 0;
}
extern "C" int dppo_debug_mma_probe(dppo_handle* h, int grid, int mode, int iters, int N, int depth, long long* out_host) {
    if (!h || !out_host || grid < 1 || grid > 1024 || depth < 0 || depth > 31) DPPO_FAIL(-1, "dppo_debug_mma_probe: bad arguments");
    CUDA_TRY(cudaSetDevice(h->device));
    if (!tc_shapes_ok(h)) DPPO_FAIL(-7, "tensor path unavailable");
    CUtensorMap wm;
    DPPO_TRY(tc::make_map(&wm, h->tc->net[DPPO_NET_ACTOR].w1, h->g.H, h->g.H, h->g.H, fc::WK, 64));      // four [32 k][64 n] boxes fill one 16 KB probe stage
    long long* d = nullptr;
    CUDA_TRY(cudaMalloc(&d, (size_t)grid * 2 * sizeof(long long)));
    CUDA_TRY(cudaMemset(d, 0, (size_t)grid * 2 * sizeof(long long)));
    const int smem = 16384 * 5 + 1024 + 256;
    CUDA_TRY(cudaFuncSetAttribute(fc::mma_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    fc::mma_probe_kernel<<<grid, 128, smem>>>(wm, mode, iters, N, depth, d);
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(out_host, d, (size_t)grid * 2 * sizeof(long long), cudaMemcpyDeviceToHost));
    cudaFree(d);
    return 0;
}
extern "C" int dppo_force_path(dppo_handle* h, int path) { if (!h) return -1; h->force_path = path; return 0; }

extern "C" int dppo_debug_tc_gemm(dppo_handle* h, const void* A, int a_mn, int64_t lda, const void* A2, int64_t lda2, int K2,
                                  const void* B, int b_mn, int64_t ldb, int M, int N, int K, int splits,
                                  const float* bias, int act, float* out_f32, void* out_bf16, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st;
    tc::Gemm g; memset(&g, 0, sizeof(g));
    g.A = tc::Operand{(const __nv_bfloat16*)A, a_mn != 0, M, K, lda};
    if (A2) g.A2 = tc::Operand{(const __nv_bfloat16*)A2, a_mn != 0, M, K2, lda2};
    g.B = tc::Operand{(const __nv_bfloat16*)B, b_mn != 0, N, K + (A2 ? K2 : 0), ldb};
    g.M = M; g.N = N; g.splits = splits;
    g.epi.M = M; g.epi.N = N; g.epi.bias = bias; g.epi.act = act;
    g.epi.out_f32 = out_f32; g.epi.ld_f32 = N; g.epi.split_stride = (size_t)M * N;
    g.epi.out_bf16 = (__nv_bfloat16*)out_bf16; g.epi.ld_bf16 = N;
    int r = tc::launch(h, s, g);
    return r < 0 ? r : 0;
}

// f16_scale > 0: two fp16 planes of f16_scale * src (the forward operand format); else three bf16 planes
__global__ void ts_split_planes_kernel(const float* __restrict__ src, size_t n, bf16* __restrict__ p0, bf16* __restrict__ p1, bf16* __restrict__ p2, float f16_scale = 0.f) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (f16_scale > 0.f) ts::split_f16(src[i] * f16_scale, p0[i], p1[i]);
    else ts::split_bf16_3(src[i], p0[i], p1[i], p2[i]);
}
extern "C" int dppo_debug_split_gemm(dppo_handle* h, const float* A, int a_mn, int64_t lda, const float* B, int b_mn, int64_t ldb,
                                     int M, int N, int K, int splits, int planes, float* out_f32, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st;
    if (!A || !B || !out_f32 || M < 1 || N < 1 || K < 1 || planes < 2 || planes > 4) DPPO_FAIL(-1, "dppo_debug_split_gemm: bad arguments");
    const bool f16 = planes == 4;          // two fp16 planes per operand, B scaled, two accumulators
    const size_t na = (((size_t)(a_mn ? K : M) * lda) + 7) & ~(size_t)7, nb = (((size_t)(b_mn ? K : N) * ldb) + 7) & ~(size_t)7;
    bf16* buf = nullptr;
    CUDA_TRY(cudaMalloc(&buf, 3 * (na + nb) * sizeof(bf16)));
    bf16* bb = buf + 3 * na;
    ts_split_planes_kernel<<<nblk((size_t)(a_mn ? K : M) * lda, 256), 256, 0, s>>>(A, (size_t)(a_mn ? K : M) * lda, buf, buf + na, buf + 2 * na, f16 ? 1.f : 0.f); KLAUNCH(h);
    ts_split_planes_kernel<<<nblk((size_t)(b_mn ? K : N) * ldb, 256), 256, 0, s>>>(B, (size_t)(b_mn ? K : N) * ldb, bb, bb + nb, bb + 2 * nb, f16 ? ts::F16_WSCALE : 0.f); KLAUNCH(h);
    ts::Gemm g; memset(&g, 0, sizeof(g));
    g.A = ts::Operand{{buf, buf + na, buf + 2 * na}, a_mn != 0, M, K, lda};
    g.B = ts::Operand{{bb, bb + nb, bb + 2 * nb}, b_mn != 0, N, K, ldb};
    g.M = M; g.N = N; g.splits = splits; g.planes = f16 ? 2 : planes;
    if (f16) { g.f16 = 1; g.dual = 1; g.epi.scale = 1.0f / ts::F16_WSCALE; }
    g.epi.M = M; g.epi.N = N; g.epi.out_f32 = out_f32; g.epi.ld_f32 = N; g.epi.split_stride = (size_t)M * N;
    int r = ts::launch(h, s, g);
    cudaStreamSynchronize(s);
    cudaFree(buf);
    return r < 0 ? r : 0;
}

__global__ void ts_sum_planes_kernel(const bf16* __restrict__ p0, const bf16* __restrict__ p1, const bf16* __restrict__ p2, size_t n, float* __restrict__ out, int f16 = 0) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (f16) out[i] = ts::f16_plane_value(p0[i]) + ts::f16_plane_value(p1[i]);
    else out[i] = __bfloat162float(p0[i]) + __bfloat162float(p1[i]) + (p2 ? __bfloat162float(p2[i]) : 0.f);
}
extern "C" int dppo_debug_pair_gemm(dppo_handle* h, const float* A, int64_t lda, const float* B, int b_mn, int64_t ldb,
                                    int M, int N, int K, int planes, const float* bias, int act, float* out_f32, uint32_t* mask_out, dppo_stream_t st) {
    ENTER(h); cudaStream_t s = (cudaStream_t)st;
    if (!A || !B || !out_f32 || M < 1 || N < 64 || (N % 64) || K < 1 || planes < 2 || planes > 4) DPPO_FAIL(-1, "dppo_debug_pair_gemm: bad arguments");
    const bool f16 = planes == 4;          // fp16 planes in and out, B scaled, two accumulators
    const size_t na = (((size_t)M * lda) + 7) & ~(size_t)7, nb = (((size_t)(b_mn ? K : N) * ldb) + 7) & ~(size_t)7, no = (((size_t)M * N) + 7) & ~(size_t)7;
    bf16* buf = nullptr;
    CUDA_TRY(cudaMalloc(&buf, 3 * (na + nb + no) * sizeof(bf16)));
    bf16* bb = buf + 3 * na; bf16* ob = bb + 3 * nb;
    ts_split_planes_kernel<<<nblk((size_t)M * lda, 256), 256, 0, s>>>(A, (size_t)M * lda, buf, buf + na, buf + 2 * na, f16 ? 1.f : 0.f); KLAUNCH(h);
    ts_split_planes_kernel<<<nblk((size_t)(b_mn ? K : N) * ldb, 256), 256, 0, s>>>(B, (size_t)(b_mn ? K : N) * ldb, bb, bb + nb, bb + 2 * nb, f16 ? ts::F16_WSCALE : 0.f); KLAUNCH(h);
    tsp::Gemm g; memset(&g, 0, sizeof(g));
    g.A = ts::Operand{{buf, buf + na, buf + 2 * na}, false, M, K, lda};
    g.B = ts::Operand{{bb, bb + nb, bb + 2 * nb}, b_mn != 0, N, K, ldb};
    g.M = M; g.N = N; g.planes = f16 ? 2 : planes; g.dual = (planes == 3 || f16) ? 1 : 0;
    if (f16) { g.f16 = 1; g.epi.scale = 1.0f / ts::F16_WSCALE; }
    g.out[0] = ob; g.out[1] = ob + no; g.out[2] = ob + 2 * no; g.ld_out = N;
    g.epi.M = M; g.epi.N = N; g.epi.out_planes = f16 ? 2 : planes; g.epi.bias = bias; g.epi.act = act;
    if (mask_out) { g.epi.mask_out = mask_out; g.epi.ldm = N / 32; }
    int r = tsp::launch(h, s, g);
    if (r == 0) { ts_sum_planes_kernel<<<nblk((size_t)M * N, 256), 256, 0, s>>>(ob, ob + no, planes == 3 ? ob + 2 * no : nullptr, (size_t)M * N, out_f32, f16 ? 1 : 0); KLAUNCH(h); }
    cudaStreamSynchronize(s);
    cudaFree(buf);
    return r;
}
