// C ABI of the Harmony engine (include/harmony_b200.h): context, uploads, stage launches.
// Host-side orchestration only -- all arithmetic on cells happens in hmy_round.cuh /
// hmy_ridge.cuh.  Built in-tree by __graft_entry__.build() with
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>
#include <thread>
#include <mutex>
#include <condition_variable>
#include <functional>
#include <sys/mman.h>
#include <unistd.h>
#include <chrono>
#include <cstdlib>

#define HMY_NONTEMPLATE_KERNELS 1
#include "../../include/harmony_b200.h"
#include "hmy_common.cuh"
#include "hmy_round.cuh"
#include "hmy_round_mma.cuh"
#include "hmy_round_tc5.cuh"
#include "hmy_ridge.cuh"
#include "hmy_ridge_mma.cuh"
#include "hmy_kmeans_init.cuh"

#define HMY_VERSION "harmony_b200 0.1.0 (sm_100a)"

static thread_local std::string g_create_error;

struct EventPair { cudaEvent_t a, b; };

struct hmy_ctx {
    HmyDev st{};
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    std::vector<int> levels, level_off;
    int KPT = 0, JPW = 0;
    int WN = 1, NT = 0, round_threads = HMY_THREADS;
    bool use_mma = false, want_mma = true, ridge_mma = false, want_ridge_mma = true;
    float zscale = 1.f;
    int force_wn = 0;
    // tcgen05 / tensor-memory round kernel (hmy_round_tc5.cuh): the single-GPU persistent path where its shape
    // limits hold.  want_tc5: -1 auto (default), 0 off, 1 required (unsupported shapes fail)
    int want_tc5 = -1;
    bool tc5_ok = false;                    // shape supported (decided in plan_round)
    bool legacy_ok = true;                  // the mma.sync / SIMT round kernels fit (their K x B tables live in shared memory)
    bool t5_state = false;                  // the device tables (running O, removed sums) were produced by that kernel
    int tc5_nc = 0, smem_tc5 = 0, G_tc5 = 0;
    const void* fn_tc5 = nullptr; const void* fn_tc5_multi = nullptr;
    unsigned int x5_seq = 0;                // LL sequence number of the last multi-GPU launch of that kernel
    unsigned char* blkbuf[2] = {nullptr, nullptr};      // block of every cell: round r in blkbuf[r & 1]
    float* t5_told[2] = {nullptr, nullptr}; int told_cur = 0;     // [nblk][B][K] removed sums | [nblk][K] their row sums
    float* t5_dnew = nullptr;                                      // [nblk][B][K] re-added sums | [nblk][K] row sums
    size_t t5_table_floats = 0;
    double* t5_rsum[2] = {nullptr, nullptr}; int rsum_cur = 0;
    unsigned long long bar_count64 = 0;     // host mirror of the device grid-barrier counter
    long long n_assigned = 0, n_done = 0;   // rounds (since init) with a block assignment / executed
    int write_r = 1; bool r_valid = true;   // R rows in HBM are those of the last stage
    long long dma_direct = 0;               // transfers that went straight from / to the caller's page-locked array
    double* objring = nullptr;              // [16][4] objective sums of the last stages (tc5 path), [16][2] all-rank sums behind them
    long long stages_launched = 0;          // tc5 stages launched so far (ring slot = stages_launched % 16)
    int G = 0, sms = 0;
    int smem_round = 0, smem_mom = 0, smem_apply = 0, smem_solve = 0;
    int grid_ridge = 0, grid_mom = 0, ridge_threads = HMY_THREADS;
    bool persistent = true;
    bool have_data = false, have_params = false, have_init = false;
    unsigned long long seed = 0x243F6A8885A308D3ull;
    unsigned int round_counter = 0, gen = 0;
    double block_size = 0.05;
    // kernels bound to the (KPT, JPW) instantiation
    const void* fn_round = nullptr; const void* fn_stage = nullptr; const void* fn_round_fused = nullptr;
    const void* fn_mom = nullptr; const void* fn_apply = nullptr;
    // device buffers
    std::vector<void*> allocs;
    float* Ybuf[2] = {nullptr, nullptr};
    int ycur = 0;            // Ybuf[ycur] feeds the next stage
    float* Ylast = nullptr;  // centroids the last finished round used (the reference's _Y)
    unsigned char* zero_round = nullptr; size_t zero_round_bytes = 0;
    unsigned char* zero_ridge = nullptr; size_t zero_ridge_bytes = 0;
    long long* d_perm = nullptr;
    int* d_cnt = nullptr; int list_chunks = 0;
    float* d_tmp = nullptr; size_t tmp_bytes = 0;
    unsigned char* h_stage[2] = {nullptr, nullptr};      // pinned bounce buffers for result reads
    cudaEvent_t ev_stage[2] = {nullptr, nullptr};
    double* h_obj = nullptr;     // pinned
    // counters / timers
    long long launches = 0, rounds = 0, ridge_passes = 0;
    bool timing = true;
    std::vector<EventPair> ev_round, ev_ridge, ev_init;
    double ms_round = 0.0, ms_ridge = 0.0, ms_init = 0.0;
    // multi-GPU
    hmy_allreduce_fn ar = nullptr; void* ar_user = nullptr;
    unsigned char* xbuf = nullptr; size_t xbytes = 0;      // this rank's exchange buffer
    std::vector<void*> xopened;                            // peers' buffers opened through IPC
    bool fused = false, force_fused_kernel = false;
    unsigned int xseq = 0;
    int rank = -1, world = 0;                              // hmy_set_rank / hmy_comm_attach (host side only)
    double* kmi_agree = nullptr; int kmi_agree_world = 0;  // [world][HMY_KMI_AGREE] checks exchanged by hmy_kmeans_init
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            char b_[512];                                                                          \
            snprintf(b_, sizeof b_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            ctx->err = b_;                                                                         \
            return 1;                                                                              \
        }                                                                                          \
    } while (0)

#define FAIL(msg) do { ctx->err = (msg); return 1; } while (0)

template <class T>
static int dev_alloc(hmy_ctx* ctx, T** p, size_t count) {
    void* q = nullptr;
    CK(cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T)));
    ctx->allocs.push_back(q);
    *p = (T*)q;
    return 0;
}

// Each (KPT, JPW) instantiation of the streaming kernels lives in its own translation unit
// (hmy_inst.cu, compiled once per pair so the build parallelises); it exports
// hmy_bind_<KPT>_<JPW>(fns) filling {k_round, k_round_stage, k_ridge_moments, k_ridge_apply}.
#define HMY_DECL_BIND(K_, J_) extern "C" void hmy_bind_##K_##_##J_(const void** fns);
HMY_DECL_BIND(1, 4) HMY_DECL_BIND(1, 8) HMY_DECL_BIND(1, 16)
HMY_DECL_BIND(2, 4) HMY_DECL_BIND(2, 8) HMY_DECL_BIND(2, 16)
HMY_DECL_BIND(4, 4) HMY_DECL_BIND(4, 8) HMY_DECL_BIND(4, 16)
HMY_DECL_BIND(8, 4) HMY_DECL_BIND(8, 8) HMY_DECL_BIND(8, 16)

#define HMY_DECL_BIND_MMA(N_, W_) extern "C" void hmy_bind_mma_##N_##_##W_(const void** fns);
HMY_DECL_BIND_MMA(4, 1) HMY_DECL_BIND_MMA(8, 1) HMY_DECL_BIND_MMA(14, 1) HMY_DECL_BIND_MMA(16, 1)
HMY_DECL_BIND_MMA(8, 2) HMY_DECL_BIND_MMA(14, 2) HMY_DECL_BIND_MMA(16, 2)

static inline bool use_tc5(const hmy_ctx* ctx);
static int split_zcos(hmy_ctx* ctx);
extern "C" void hmy_bind_tc5_4(const void** fns);
extern "C" void hmy_bind_tc5_7(const void** fns);
extern "C" void hmy_bind_tc5_8(const void** fns);

// tensor-core round kernels: d <= 64 and K <= 256 (everything else stays on the SIMT kernels)
static bool bind_mma(hmy_ctx* ctx) {
    const HmyDev& st = ctx->st;
    if (st.d > 64 || st.K > 256) return false;
    const int KT = (st.K + 7) / 8;
    ctx->WN = (st.K <= 128) ? 1 : 2;
    if (ctx->force_wn == 2 && KT >= 2) ctx->WN = 2;
    const int ntw = (ctx->WN == 1) ? KT : (KT + 1) / 2;
    const void* f[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    if (ctx->WN == 1) {
        if (ntw <= 4) { hmy_bind_mma_4_1(f); ctx->NT = 4; } else if (ntw <= 8) { hmy_bind_mma_8_1(f); ctx->NT = 8; }
        else if (ntw <= 14) { hmy_bind_mma_14_1(f); ctx->NT = 14; } else { hmy_bind_mma_16_1(f); ctx->NT = 16; }
    } else {
        if (ntw <= 8) { hmy_bind_mma_8_2(f); ctx->NT = 8; } else if (ntw <= 14) { hmy_bind_mma_14_2(f); ctx->NT = 14; }
        else { hmy_bind_mma_16_2(f); ctx->NT = 16; }
    }
    ctx->fn_round = f[0]; ctx->fn_stage = f[1]; ctx->fn_round_fused = f[4];
    ctx->round_threads = 128 * ctx->WN;
    ctx->use_mma = true;
    ctx->ridge_mma = false;
    if (st.d <= 63 && ctx->want_ridge_mma) {
        ctx->fn_mom = f[2]; ctx->fn_apply = f[3];
        ctx->ridge_mma = true;
    }
    return true;
}

static bool bind_for(hmy_ctx* ctx) {
    const void* f[4] = {nullptr, nullptr, nullptr, nullptr};
    switch (ctx->KPT * 100 + ctx->JPW) {
        case 104: hmy_bind_1_4(f); break;   case 108: hmy_bind_1_8(f); break;   case 116: hmy_bind_1_16(f); break;
        case 204: hmy_bind_2_4(f); break;   case 208: hmy_bind_2_8(f); break;   case 216: hmy_bind_2_16(f); break;
        case 404: hmy_bind_4_4(f); break;   case 408: hmy_bind_4_8(f); break;   case 416: hmy_bind_4_16(f); break;
        case 804: hmy_bind_8_4(f); break;   case 808: hmy_bind_8_8(f); break;   case 816: hmy_bind_8_16(f); break;
        default: return false;
    }
    ctx->fn_round = f[0]; ctx->fn_stage = f[1]; ctx->fn_mom = f[2]; ctx->fn_apply = f[3];
    return true;
}

extern "C" const char* hmy_version(void) { return HMY_VERSION; }

// failure channel of the context-free entry points in other translation units (hmy_lisi.cu)
extern "C" void harmony_b200_set_global_error(const char* msg) { g_create_error = msg ? msg : ""; }

extern "C" const char* hmy_last_error(const hmy_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

static int create_impl(hmy_ctx* ctx, int device, int64_t n_local, int64_t n_global, int64_t cell_offset,
                       int d, int K, int V, const int32_t* levels_per_var) {
    HmyDev& st = ctx->st;
    if (n_local < 1 || n_local > 2000000000LL) FAIL("n_local out of range (1 .. 2e9 cells per rank)");
    if (n_global < n_local || cell_offset < 0 || cell_offset + n_local > n_global) FAIL("cell range outside n_global");
    if (d < 1 || d > 128) FAIL("d must be in 1..128");
    if (K < 2 || K > 256) FAIL("K (nclust) must be in 2..256");
    if (V < 1 || V > HMY_MAX_V) FAIL("number of batch covariates must be in 1..8");
    ctx->device = device;
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    ctx->sms = prop.multiProcessorCount;
    int B = 0;
    for (int v = 0; v < V; ++v) {
        if (levels_per_var[v] < 1) FAIL("every covariate needs at least one level");
        ctx->levels.push_back(levels_per_var[v]);
        ctx->level_off.push_back(B);
        B += levels_per_var[v];
    }
    st.N = n_local; st.Nglobal = n_global; st.cell_offset = cell_offset;
    st.d = d; st.dp = (d + 3) & ~3; st.K = K; st.Kp = (K + 3) & ~3;
    ctx->KPT = (K <= 32) ? 1 : (K <= 64) ? 2 : (K <= 128) ? 4 : 8;
    ctx->JPW = (st.dp <= 32) ? 4 : (st.dp <= 64) ? 8 : 16;
    st.KS = 32 * ctx->KPT;
    st.V = V; st.B = B; st.lev0 = levels_per_var[0];
    if (!bind_for(ctx)) FAIL("no kernel instantiation for this (K, d)");
    // state
    if (dev_alloc(ctx, &st.Zorig, (size_t)st.N * st.dp)) return 1;
    if (dev_alloc(ctx, &st.Zcos, (size_t)st.N * st.dp)) return 1;
    if (dev_alloc(ctx, &st.Zcorr, (size_t)st.N * st.dp)) return 1;
    if (dev_alloc(ctx, &st.R, (size_t)st.N * st.Kp)) return 1;
    if (dev_alloc(ctx, &st.combo, (size_t)st.N)) return 1;
    if (dev_alloc(ctx, &st.order, (size_t)st.N)) return 1;
    if (dev_alloc(ctx, &st.pos_of, (size_t)st.N)) return 1;
    if (dev_alloc(ctx, &st.blk, (size_t)st.N)) return 1;
    if (dev_alloc(ctx, &st.list, (size_t)st.N)) return 1;
    if (dev_alloc(ctx, &ctx->Ybuf[0], (size_t)K * st.dp)) return 1;
    if (dev_alloc(ctx, &ctx->Ybuf[1], (size_t)K * st.dp)) return 1;
    if (dev_alloc(ctx, &st.P, (size_t)B * K)) return 1;
    if (dev_alloc(ctx, &st.O, (size_t)B * K)) return 1;
    if (dev_alloc(ctx, &st.Orun, (size_t)B * K)) return 1;
    if (dev_alloc(ctx, &st.obj_out, 4)) return 1;
    if (dev_alloc(ctx, &st.Pr_b, (size_t)B)) return 1;
    if (dev_alloc(ctx, &st.theta, (size_t)B)) return 1;
    if (dev_alloc(ctx, &st.sigma, (size_t)K)) return 1;
    if (dev_alloc(ctx, &st.lamb, (size_t)B + 1)) return 1;
    if (dev_alloc(ctx, &st.W, (size_t)B * K * st.dp)) return 1;
    if (dev_alloc(ctx, &st.wmax, 4)) return 1;
    if (dev_alloc(ctx, &st.bar_count, 2)) return 1;
    st.bar_gen = st.bar_count + 1;
    CK(cudaMemset(st.bar_count, 0, 2 * sizeof(unsigned int)));
    if (dev_alloc(ctx, &st.bar64, 1)) return 1;
    CK(cudaMemset(st.bar64, 0, sizeof(unsigned long long)));
    if (K <= 128 && d <= 64) {
        // operands of the tensor-memory round kernel: pre-split Z_cos rows, annotated lists, two block-id buffers
        const int dt = (d + 15) / 16;
        if (dev_alloc(ctx, &st.Zs16, (size_t)st.N * 32 * dt)) return 1;
        if (dev_alloc(ctx, &st.list2, (size_t)st.N)) return 1;
        if (dev_alloc(ctx, &ctx->blkbuf[0], (size_t)st.N)) return 1;
        if (dev_alloc(ctx, &ctx->blkbuf[1], (size_t)st.N)) return 1;
    }
    CK(cudaMemset(st.O, 0, (size_t)B * K * sizeof(double)));
    CK(cudaMemset(st.W, 0, (size_t)B * K * st.dp * sizeof(float)));
    // ridge accumulators in one zeroable block: Gram | Mom
    {
        const size_t nG = (size_t)K * (B + 1) * (B + 1), nM = (size_t)(B + 1) * K * st.dp;
        ctx->zero_ridge_bytes = (nG + nM) * sizeof(double);
        if (dev_alloc(ctx, &ctx->zero_ridge, ctx->zero_ridge_bytes)) return 1;
        st.Gram = (double*)ctx->zero_ridge; st.Mom = st.Gram + nG;
    }
    CK(cudaMallocHost((void**)&ctx->h_obj, 4 * sizeof(double)));
    st.Yhat = ctx->Ybuf[0]; st.Ynext = ctx->Ybuf[1]; ctx->Ylast = ctx->Ybuf[0];
    CK(cudaMemset(ctx->Ybuf[0], 0, (size_t)K * st.dp * sizeof(float)));
    CK(cudaMemset(ctx->Ybuf[1], 0, (size_t)K * st.dp * sizeof(float)));
    // ridge launch shapes
    ctx->smem_mom = ridge_smem_plan(K, st.KS, ctx->JPW, false).total;
    ctx->smem_apply = ridge_smem_plan(K, st.KS, ctx->JPW, true).total;
    {
        const size_t per = (size_t)(B + 1) * (B + 1 + d) + (B + 1);
        if (per * sizeof(double) > 200 * 1024) {
            // many batch levels: the K augmented systems go to a global work area instead of shared memory
            if (dev_alloc(ctx, &st.solve_scratch, (size_t)K * per)) return 1;
            ctx->smem_solve = 0;
        } else {
            ctx->smem_solve = (int)(per * sizeof(double));
            CK(cudaFuncSetAttribute((const void*)k_ridge_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_solve));
        }
    }
    return 0;
}

extern "C" int hmy_create(hmy_ctx** out, int device, int64_t n_local, int64_t n_global, int64_t cell_offset,
                          int d, int K, int V, const int32_t* levels_per_var) {
    if (!out) { g_create_error = "hmy_create: out is NULL"; return 1; }
    *out = nullptr;
    hmy_ctx* ctx = new hmy_ctx();
    if (create_impl(ctx, device, n_local, n_global, cell_offset, d, K, V, levels_per_var)) {
        g_create_error = ctx->err;
        hmy_destroy(ctx);
        return 1;
    }
    *out = ctx;
    return 0;
}

extern "C" void hmy_destroy(hmy_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (void* p : ctx->xopened) cudaIpcCloseMemHandle(p);
    if (ctx->xbuf) cudaFree(ctx->xbuf);
    for (void* p : ctx->allocs) cudaFree(p);
    if (ctx->d_perm) cudaFree(ctx->d_perm);
    if (ctx->d_tmp) cudaFree(ctx->d_tmp);
    if (ctx->h_obj) cudaFreeHost(ctx->h_obj);
    for (int i = 0; i < 2; ++i) { if (ctx->h_stage[i]) cudaFreeHost(ctx->h_stage[i]); if (ctx->ev_stage[i]) cudaEventDestroy(ctx->ev_stage[i]); }
    for (auto& e : ctx->ev_round) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
    for (auto& e : ctx->ev_ridge) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
    for (auto& e : ctx->ev_init) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
    delete ctx;
}

extern "C" int hmy_set_stream(hmy_ctx* ctx, void* cuda_stream) {
    ctx->stream = (cudaStream_t)cuda_stream;
    return 0;
}

// round launch shape: depends on nblk (shared-memory plan), so fixed once block_size is known
static int plan_round(hmy_ctx* ctx) {
    HmyDev& st = ctx->st;
    const int nblk = (int)std::ceil(1.0 / (double)ctx->block_size);          // harmony.py:474
    if (nblk < 1 || nblk > HMY_MAX_NBLK) FAIL("block_size gives an unsupported number of blocks (1..250)");
    st.nblk = nblk;
    st.cpb = (long long)((double)st.Nglobal * (double)ctx->block_size);      // harmony.py:475
    if (!bind_for(ctx)) FAIL("no kernel instantiation for this (K, d)");
    ctx->use_mma = false; ctx->round_threads = HMY_THREADS;
    if (ctx->want_mma) bind_mma(ctx);
    ctx->smem_round = ctx->use_mma ? mma_smem_plan(st.d, st.K, st.KS, st.B, st.V, nblk, ctx->WN, ctx->NT).total
                                   : round_smem_plan(st.dp, st.KS, st.B, st.V, nblk, ctx->JPW).total;
    // these kernels keep two K x B tables per CTA in shared memory: with hundreds of batch levels they do not fit, and
    // only the tensor-memory kernel (no K x B tables on chip) can run such a problem -- decided when a stage is launched
    ctx->legacy_ok = ctx->smem_round <= 227 * 1024;
    ctx->G = ctx->sms;
    if (ctx->legacy_ok) {
        CK(cudaFuncSetAttribute(ctx->fn_round, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_round));
        if (ctx->use_mma) CK(cudaFuncSetAttribute(ctx->fn_round_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_round));
        CK(cudaFuncSetAttribute(ctx->fn_stage, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_round));
        int nb = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, ctx->fn_round, ctx->round_threads, ctx->smem_round));
        if (nb < 1) FAIL("round kernel does not fit on an SM");
        ctx->G = nb * ctx->sms;
    }
    ctx->tc5_ok = false;
    if (ctx->want_tc5 != 0) {
        const bool shape = st.K <= 128 && st.d <= 64 && nblk <= 32 && st.B <= 65535 && st.Zs16 != nullptr;
        // option tc5 = 1 asks for this kernel: unsupported shapes fail loudly, there is no silent fallback then
        if (!shape && ctx->want_tc5 == 1)
            FAIL("option tc5: the tensor-memory round kernel needs K <= 128, d <= 64 and at most 32 blocks");
        if (shape) {
            const void* f[2] = {nullptr, nullptr};
            if (st.K <= 64) { hmy_bind_tc5_4(f); ctx->tc5_nc = 4; } else if (st.K <= 112) { hmy_bind_tc5_7(f); ctx->tc5_nc = 7; } else { hmy_bind_tc5_8(f); ctx->tc5_nc = 8; }
            ctx->fn_tc5 = f[0]; ctx->fn_tc5_multi = f[1];
            ctx->smem_tc5 = t5_smem_bytes(ctx->tc5_nc);
            CK(cudaFuncSetAttribute(ctx->fn_tc5, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_tc5));
            CK(cudaFuncSetAttribute(ctx->fn_tc5_multi, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_tc5));
            int nt5 = 0;
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nt5, ctx->fn_tc5, T5_THREADS, ctx->smem_tc5));
            if (nt5 < 1) FAIL("tensor-memory round kernel does not fit on an SM");
            ctx->G_tc5 = ctx->sms;            // one CTA per SM: it owns the SM's tensor memory
            ctx->t5_table_floats = (size_t)nblk * st.B * st.K + (size_t)nblk * st.K;
            for (int i = 0; i < 2; ++i) {
                if (dev_alloc(ctx, &ctx->t5_told[i], ctx->t5_table_floats)) return 1;
                if (dev_alloc(ctx, &ctx->t5_rsum[i], (size_t)st.K)) return 1;
            }
            if (dev_alloc(ctx, &ctx->t5_dnew, ctx->t5_table_floats)) return 1;
            if (dev_alloc(ctx, &ctx->objring, (size_t)16 * 6)) return 1;
            ctx->tc5_ok = true;
        }
    }
    // per-round zero block: Told | Dnew | Yacc is separate (ridge also uses it) | obj
    const size_t nT = (size_t)nblk * st.B * st.K;
    ctx->zero_round_bytes = 2 * nT * sizeof(float) + (4 + (size_t)st.B * st.K + (size_t)st.K * st.dp) * sizeof(double);
    ctx->zero_round_bytes = (ctx->zero_round_bytes + 7) & ~(size_t)7;
    if (dev_alloc(ctx, &ctx->zero_round, ctx->zero_round_bytes + 8)) return 1;
    st.obj = (double*)ctx->zero_round;                      // 8-byte aligned at the front
    st.Ofresh = st.obj + 4;
    st.Yacc = st.Ofresh + (size_t)st.B * st.K;              // obj | Ofresh | Yacc: one exchange / all-reduce
    st.Told = (float*)(st.Yacc + (size_t)st.K * st.dp); st.Dnew = st.Told + nT;
    if (dev_alloc(ctx, &st.blk_start, (size_t)nblk + 1)) return 1;
    ctx->list_chunks = std::min(4 * ctx->sms, 32 * HMY_SCAN_PER_LANE);
    {
        const size_t sm = ((size_t)nblk * HMY_LIST_THREADS + nblk) * sizeof(unsigned int);
        if (sm > 200 * 1024) FAIL("block_size gives too many blocks for the list builder");
        CK(cudaFuncSetAttribute((const void*)k_block_lists, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    }
    if (dev_alloc(ctx, &ctx->d_cnt, (size_t)ctx->list_chunks * nblk)) return 1;
    if (ctx->ridge_mma) {
        ctx->smem_mom = ridge_mma_plan(st.d, ctx->WN, ctx->NT, false).total;
        ctx->smem_apply = ridge_mma_plan(st.d, ctx->WN, ctx->NT, true).total;
        if (ctx->smem_apply > 227 * 1024) FAIL("ridge apply kernel needs more than 227 KB of shared memory");
    } else {
        ctx->smem_mom = ridge_smem_plan(st.K, st.KS, ctx->JPW, false).total;
        ctx->smem_apply = ridge_smem_plan(st.K, st.KS, ctx->JPW, true).total;
    }
    ctx->ridge_threads = ctx->ridge_mma ? 128 * ctx->WN : HMY_THREADS;
    CK(cudaFuncSetAttribute(ctx->fn_mom, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_mom));
    CK(cudaFuncSetAttribute(ctx->fn_apply, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_apply));
    int nbr = 0, nbm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nbr, ctx->fn_apply, ctx->ridge_threads, ctx->smem_apply));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nbm, ctx->fn_mom, ctx->ridge_threads, ctx->smem_mom));
    ctx->grid_ridge = std::max(1, nbr) * ctx->sms;
    ctx->grid_mom = std::max(1, nbm) * ctx->sms;
    return 0;
}

extern "C" int hmy_set_params(hmy_ctx* ctx, const float* Pr_b, const float* theta, const float* sigma,
                              const float* lamb, int lambda_estimation, float alpha, double block_size) {
    HmyDev& st = ctx->st;
    CK(cudaSetDevice(ctx->device));
    if (ctx->have_params) FAIL("hmy_set_params may be called once per context");
    if (!(block_size > 0.0) || block_size > 1.0) FAIL("block_size must be in (0, 1]");
    ctx->block_size = block_size;
    CK(cudaMemcpy(st.Pr_b, Pr_b, st.B * sizeof(float), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(st.theta, theta, st.B * sizeof(float), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(st.sigma, sigma, st.K * sizeof(float), cudaMemcpyHostToDevice));
    std::vector<float> l(st.B + 1, 0.f);
    if (!lambda_estimation) { if (!lamb) FAIL("lamb is NULL"); std::copy(lamb, lamb + st.B + 1, l.begin()); }
    CK(cudaMemcpy(st.lamb, l.data(), (st.B + 1) * sizeof(float), cudaMemcpyHostToDevice));
    st.sigma_uniform = 1; st.sigma_u = sigma[0];
    for (int k = 1; k < st.K; ++k) if (sigma[k] != sigma[0]) st.sigma_uniform = 0;
    st.lambda_estimation = lambda_estimation ? 1 : 0;
    st.alpha = alpha;
    if (plan_round(ctx)) return 1;
    ctx->have_params = true;
    return 0;
}

// ---- host-side helpers of the upload / download paths ------------------------------------------------------------
static int host_threads() { const unsigned hc = std::thread::hardware_concurrency(); return (int)std::max(1u, std::min(16u, hc ? hc : 4u)); }
#define HMY_STAGE_CHUNK ((size_t)16u << 20)

// A few persistent host threads for the copies and index builds of the upload / download paths (creating 16
// threads per 16 MB chunk cost more than the copy itself: 200 MB moved at 7 GB/s).  Process-wide, created on first use.
class HostPool {
  public:
    explicit HostPool(int n) : n_(n) { for (int t = 1; t < n; ++t) th_.emplace_back([this, t]() { loop(t); }); }
    ~HostPool() { { std::lock_guard<std::mutex> g(m_); stop_ = true; } cv_.notify_all(); for (auto& x : th_) x.join(); }
    int size() const { return n_; }
    void run(const std::function<void(int)>& f) {          // f(t) for t in [0, n), t = 0 on the caller; returns when all are done
        if (n_ == 1) { f(0); return; }
        std::lock_guard<std::mutex> one_caller(run_m_);      // contexts driven from different host threads share the pool
        { std::lock_guard<std::mutex> g(m_); job_ = &f; pending_ = n_ - 1; ++gen_; }
        cv_.notify_all();
        f(0);
        std::unique_lock<std::mutex> g(m_);
        done_.wait(g, [this]() { return pending_ == 0; });
        job_ = nullptr;
    }
  private:
    void loop(int t) {
        unsigned long long seen = 0;
        for (;;) {
            const std::function<void(int)>* f;
            { std::unique_lock<std::mutex> g(m_); cv_.wait(g, [&]() { return stop_ || gen_ != seen; }); if (stop_) return; seen = gen_; f = job_; }
            (*f)(t);
            { std::lock_guard<std::mutex> g(m_); if (--pending_ == 0) done_.notify_one(); }
        }
    }
    int n_; std::vector<std::thread> th_; std::mutex m_, run_m_; std::condition_variable cv_, done_;
    const std::function<void(int)>* job_ = nullptr; int pending_ = 0; unsigned long long gen_ = 0; bool stop_ = false;
};
static HostPool& host_pool() { static HostPool p(host_threads()); return p; }

// fn(t, lo, hi) over [0, n) split into contiguous ranges, one per thread (range t precedes range t + 1)
template <class F>
static void parallel_ranges(long long n, int T, F fn) {
    if (T <= 1 || n < 65536) { fn(0, 0LL, n); return; }
    HostPool& pool = host_pool();
    const int P = pool.size();
    pool.run([&](int t) { fn(t, n * t / P, n * (t + 1) / P); });
}

static int ensure_stage(hmy_ctx* ctx) {
    constexpr size_t CHUNK = HMY_STAGE_CHUNK;
    if (!ctx->h_stage[0])
        for (int i = 0; i < 2; ++i) { CK(cudaMallocHost((void**)&ctx->h_stage[i], CHUNK)); CK(cudaEventCreateWithFlags(&ctx->ev_stage[i], cudaEventDisableTiming)); }
    return 0;
}

// true when p lies in page-locked host memory the CUDA runtime knows (hmy_host_alloc, cudaHostAlloc, cudaHostRegister,
// torch pinned tensors): such arrays move by DMA alone
static bool host_is_pinned(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

extern "C" void* hmy_host_alloc(int device, size_t bytes) {
    void* p = nullptr;
    if (cudaSetDevice(device) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
    return p;
}
extern "C" void hmy_host_free(void* p) {
    if (p && cudaFreeHost(p) != cudaSuccess) (void)cudaGetLastError();
}

// pageable host memory -> device through the two pinned bounce buffers: the host copy of chunk i + 1 (spread over
// threads) overlaps the DMA of chunk i (a plain cudaMemcpy from pageable memory stages single-threaded inside the driver)
static int h2d_staged(hmy_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes) {
    constexpr size_t CHUNK = HMY_STAGE_CHUNK;
    if (bytes >= (1u << 20) && host_is_pinned(src_host)) {
        // the caller keeps the array in page-locked memory: one DMA, no host copy (every caller of this function
        // synchronises the stream before the source can go away)
        CK(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
        ctx->dma_direct++;
        return 0;
    }
    if (ensure_stage(ctx)) return 1;
    const unsigned char* src8 = (const unsigned char*)src_host; unsigned char* dst8 = (unsigned char*)dst_dev;
    const size_t nchunk = (bytes + CHUNK - 1) / CHUNK;
    const int T = host_threads();
    for (size_t i = 0; i < nchunk; ++i) {
        const size_t off = i * CHUNK, len = std::min(CHUNK, bytes - off);
        CK(cudaEventSynchronize(ctx->ev_stage[i & 1]));          // the DMA that last used this buffer (this call or an earlier one) is done
        unsigned char* hb = ctx->h_stage[i & 1];
        parallel_ranges((long long)len, len >= (2u << 20) ? T : 1, [&](int, long long lo, long long hi) { std::memcpy(hb + lo, src8 + off + lo, (size_t)(hi - lo)); });
        CK(cudaMemcpyAsync(dst8 + off, hb, len, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaEventRecord(ctx->ev_stage[i & 1], ctx->stream));
    }
    return 0;
}

extern "C" int hmy_set_data(hmy_ctx* ctx, const float* Z_host, const int32_t* codes_host) {
    HmyDev& st = ctx->st;
    CK(cudaSetDevice(ctx->device));
    const bool tm = std::getenv("HMY_TIMING") != nullptr;
    auto t_prev = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!tm) return;
        auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[hmy_set_data] %-28s %7.2f ms\n", what, std::chrono::duration<double, std::milli>(now - t_prev).count());
        t_prev = now;
    };
    if (!Z_host || !codes_host) FAIL("hmy_set_data: NULL input");
    const long long N = st.N; const int V = st.V;
    const int T = host_threads();
    // the big upload first: it streams through the pinned buffers while the host builds the layout below.
    // R (N x Kp floats, not valid before the init assignment) is the landing area of the raw rows.
    // Landing area of the raw rows: a buffer that is not valid yet and at least N x d floats large -- R (N x Kp) or the
    // pre-split operand rows (N x 64 ceil(d / 16) bytes >= 4 d); a temporary allocation only when neither fits.
    float* raw = nullptr; float* raw_tmp = nullptr;
    if (st.Kp >= st.d) raw = st.R;
    else if (st.Zs16) raw = reinterpret_cast<float*>(st.Zs16);
    else { CK(cudaMalloc((void**)&raw_tmp, (size_t)N * st.d * sizeof(float))); raw = raw_tmp; }
    // combination key of every cell (covariate 0 most significant)
    std::vector<unsigned long long> mult(V, 1ull);
    {
        long double span = 1.0L;
        for (int v = V - 1; v >= 0; --v) { mult[v] = (unsigned long long)span; span *= ctx->levels[v]; }
        if (span > 9.0e18L) FAIL("product of covariate level counts overflows 64 bits");
    }
    std::vector<unsigned long long> key((size_t)N);
    std::vector<unsigned long long> tmax((size_t)T, 0ull);
    std::vector<int> bad((size_t)T, 0);
    parallel_ranges(N, T, [&](int t, long long lo, long long hi) {
        unsigned long long m = 0; int b = 0;
        for (long long n = lo; n < hi; ++n) {
            unsigned long long k = 0;
            for (int v = 0; v < V; ++v) {
                const int c = codes_host[(size_t)v * N + n];
                if (c < 0 || c >= ctx->levels[v]) { b = 1; continue; }
                k += (unsigned long long)c * mult[v];
            }
            key[n] = k; m = std::max(m, k);
        }
        tmax[t] = m; bad[t] = b;
    });
    for (int t = 0; t < T; ++t) if (bad[t]) FAIL("level code out of range");
    const unsigned long long kmax = *std::max_element(tmax.begin(), tmax.end());
    // stable sort of the cells by combination key: parallel counting sort when the key range is small (the usual case:
    // a handful of batch covariates), comparison sort otherwise
    std::vector<int> order((size_t)N);
    if (kmax < (1ull << 16)) {
        const size_t nk = (size_t)kmax + 1;
        std::vector<long long> cnt((size_t)T * nk, 0);
        parallel_ranges(N, T, [&](int t, long long lo, long long hi) { long long* c = &cnt[(size_t)t * nk]; for (long long n = lo; n < hi; ++n) c[key[n]]++; });
        long long run = 0;                                             // exclusive scan in (key, thread) order: stable
        for (size_t k = 0; k < nk; ++k) for (int t = 0; t < T; ++t) { const long long c = cnt[(size_t)t * nk + k]; cnt[(size_t)t * nk + k] = run; run += c; }
        parallel_ranges(N, T, [&](int t, long long lo, long long hi) { long long* c = &cnt[(size_t)t * nk]; for (long long n = lo; n < hi; ++n) order[(size_t)c[key[n]]++] = (int)n; });
    } else if (kmax < (1ull << 22)) {
        std::vector<long long> cnt((size_t)kmax + 2, 0);
        for (long long n = 0; n < N; ++n) cnt[key[n] + 1]++;
        for (size_t i = 1; i < cnt.size(); ++i) cnt[i] += cnt[i - 1];
        for (long long n = 0; n < N; ++n) order[(size_t)cnt[key[n]]++] = (int)n;
    } else {
        std::iota(order.begin(), order.end(), 0);
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return key[a] < key[b]; });
    }
    lap("keys + counting sort");
    if (h2d_staged(ctx, raw, Z_host, (size_t)N * st.d * sizeof(float))) return 1;
    lap("H2D of Z (staged, async)");
    // combination id of every stored position: boundaries where the key changes, then a prefix count
    std::vector<int> pos_of((size_t)N), combo((size_t)N), combo_lev;
    std::vector<long long> combo_start;
    {
        std::vector<int> nb((size_t)T + 1, 0);
        parallel_ranges(N, T, [&](int t, long long lo, long long hi) {
            int c = 0;
            for (long long p = lo; p < hi; ++p) { pos_of[order[p]] = (int)p; if (p == 0 || key[order[p]] != key[order[p - 1]]) ++c; }
            nb[t + 1] = c;
        });
        for (int t = 0; t < T; ++t) nb[t + 1] += nb[t];
        const int ncombo = nb[T];
        combo_start.assign((size_t)ncombo + 1, 0);
        combo_lev.assign((size_t)ncombo * V, 0);
        const bool ran_parallel = !(T <= 1 || N < 65536);
        parallel_ranges(N, T, [&](int t, long long lo, long long hi) {
            int c = (ran_parallel ? nb[t] : 0) - 1;
            for (long long p = lo; p < hi; ++p) {
                const int src = order[p];
                if (p == 0 || key[src] != key[order[p - 1]]) {
                    ++c;
                    combo_start[c] = p;
                    for (int v = 0; v < V; ++v) combo_lev[(size_t)c * V + v] = ctx->level_off[v] + codes_host[(size_t)v * N + src];
                }
                combo[p] = c;
            }
        });
        combo_start[ncombo] = N;
        st.ncombo = ncombo;
    }
    const int ncombo = st.ncombo;
    lap("pos_of / combo tables");
    // ridge work items: <= HMY_SEG_MAX consecutive cells of one combination
    std::vector<int> seg;
    for (int c = 0; c < ncombo; ++c)
        for (long long s0 = combo_start[c]; s0 < combo_start[c + 1]; s0 += HMY_SEG_MAX) {
            seg.push_back((int)s0); seg.push_back((int)std::min<long long>(HMY_SEG_MAX, combo_start[c + 1] - s0)); seg.push_back(c);
        }
    st.nseg = (int)(seg.size() / 3);
    if (dev_alloc(ctx, &st.combo_lev, combo_lev.size())) return 1;
    if (dev_alloc(ctx, &st.combo_start, combo_start.size())) return 1;
    if (dev_alloc(ctx, &st.seg, seg.size())) return 1;
    CK(cudaMemcpyAsync(st.combo_lev, combo_lev.data(), combo_lev.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(st.combo_start, combo_start.data(), combo_start.size() * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(st.seg, seg.data(), seg.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    if (h2d_staged(ctx, st.combo, combo.data(), (size_t)N * sizeof(int))) return 1;
    if (h2d_staged(ctx, st.order, order.data(), (size_t)N * sizeof(int))) return 1;
    if (h2d_staged(ctx, st.pos_of, pos_of.data(), (size_t)N * sizeof(int))) return 1;
    lap("small uploads (async)");
    // raw rows -> sorted padded layout + Z_cos
    {
        const long long threads = N * 32;
        CK(cudaMemsetAsync(st.wmax, 0, sizeof(float), ctx->stream));        // borrowed as the |z| maximum
        k_ingest<<<(unsigned int)((threads + 255) / 256), 256, 0, ctx->stream>>>(st, raw, st.wmax);
        ctx->launches++;
        CK(cudaGetLastError());
    }
    if (split_zcos(ctx)) return 1;
    float zm = 0.f;
    CK(cudaMemcpyAsync(&zm, st.wmax, sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));          // also: the host vectors above may go out of scope now
    if (raw_tmp) cudaFree(raw_tmp);
    {   // scale of the fp16 split of Z_orig in the tensor-core ridge passes: hi part below 2^14
        int ex = 0; std::frexp(std::max(zm, 1e-30f), &ex);
        ctx->zscale = std::ldexp(1.0f, 13 - ex);
    }
    ctx->r_valid = false;                            // R served as the landing area of the upload
    lap("ingest + sync");
    ctx->have_data = true;
    return 0;
}

// ---- helpers ------------------------------------------------------------------------------
static int launch(hmy_ctx* ctx, const void* fn, dim3 grid, dim3 block, void** args, size_t smem, bool coop) {
    if (coop) CK(cudaLaunchCooperativeKernel(fn, grid, block, args, smem, ctx->stream));
    else CK(cudaLaunchKernel(fn, grid, block, args, smem, ctx->stream));
    ctx->launches++;
    return 0;
}

static int allreduce(hmy_ctx* ctx, void* p, int64_t count, int dtype) {
    if (!ctx->ar) return 0;
    if (ctx->ar(ctx->ar_user, p, count, dtype, (void*)ctx->stream)) FAIL("all-reduce callback failed");
    return 0;
}

static int timer_begin(hmy_ctx* ctx, std::vector<EventPair>& v) {
    if (!ctx->timing) return 0;
    EventPair p;
    CK(cudaEventCreate(&p.a)); CK(cudaEventCreate(&p.b));
    CK(cudaEventRecord(p.a, ctx->stream));
    v.push_back(p);
    return 0;
}
static int timer_end(hmy_ctx* ctx, std::vector<EventPair>& v) {
    if (!ctx->timing) return 0;
    CK(cudaEventRecord(v.back().b, ctx->stream));
    return 0;
}
static void timer_collect(std::vector<EventPair>& v, double& acc) {
    for (auto& p : v) {
        cudaEventSynchronize(p.b);
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) acc += ms;
        cudaEventDestroy(p.a); cudaEventDestroy(p.b);
    }
    v.clear();
}

static int fetch_obj(hmy_ctx* ctx, double obj[3]) {
    CK(cudaMemcpyAsync(ctx->h_obj, ctx->st.obj_out, 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (obj) { obj[0] = ctx->h_obj[0]; obj[1] = ctx->h_obj[1]; obj[2] = ctx->h_obj[2]; }
    return 0;
}

static void swap_centroids(hmy_ctx* ctx) {
    ctx->Ylast = ctx->Ybuf[ctx->ycur];
    ctx->ycur ^= 1;
    ctx->st.Yhat = ctx->Ybuf[ctx->ycur];
    ctx->st.Ynext = ctx->Ybuf[ctx->ycur ^ 1];
}

static int staged_tables(hmy_ctx* ctx, int what, int blk) {
    HmyDev st = ctx->st;
    void* args[] = {&st, &what, &blk};
    return launch(ctx, (const void*)k_tables, dim3(1), dim3(HMY_THREADS), args, 0, false);
}
static int staged_round(hmy_ctx* ctx, int what, int blk) {
    HmyDev st = ctx->st;
    void* args[] = {&st, &what, &blk};
    return launch(ctx, ctx->fn_stage, dim3(ctx->G), dim3(ctx->round_threads), args, ctx->smem_round, false);
}

// the persistent round kernel (cooperative launch): tensor-memory version when option "tc5" selected it
static int launch_persistent(hmy_ctx* ctx, void** args) {
    const bool fk = ctx->fused || ctx->force_fused_kernel;
    return launch(ctx, fk ? ctx->fn_round_fused : ctx->fn_round, dim3(ctx->G), dim3(ctx->round_threads), args, ctx->smem_round, true);
}


// ---- tensor-memory round kernel: host side ----------------------------------------------------------------------
// It is the path of single-GPU persistent runs whose shape it supports; sharded runs (all-reduce callback or
// peer exchange) and launch-per-block mode stay on the mma.sync / SIMT kernels.
static inline bool use_tc5(const hmy_ctx* ctx) {
    // sharded runs: with the peer exchange attached (fused) and exact per-block exchange only; the staged all-reduce
    // mode and the "relaxed" one-exchange-per-round variant stay on the mma.sync kernel
    return ctx->tc5_ok && ctx->persistent && (!ctx->ar || ctx->fused) && !(ctx->fused && ctx->st.xrelaxed);
}

static int split_zcos(hmy_ctx* ctx) {
    HmyDev& st = ctx->st;
    if (!st.Zs16) return 0;
    const long long threads = st.N * 8 * ((st.d + 15) / 16);
    k_split_zcos<<<(unsigned int)((threads + 255) / 256), 256, 0, ctx->stream>>>(st);
    ctx->launches++;
    CK(cudaGetLastError());
    return 0;
}

// block of every cell in round `round` (since init) -> blkbuf[round & 1]  (harmony.py:471-475, :483-484)
static int assign_round(hmy_ctx* ctx, const int64_t* perm_host, long long round) {
    HmyDev s = ctx->st;
    s.blk = ctx->blkbuf[round & 1];
    if (perm_host) {
        if (!ctx->d_perm) CK(cudaMalloc((void**)&ctx->d_perm, (size_t)s.Nglobal * sizeof(long long)));
        CK(cudaMemcpyAsync(ctx->d_perm, perm_host, (size_t)s.Nglobal * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
        k_assign_from_perm<<<(unsigned int)((s.Nglobal + 255) / 256), 256, 0, ctx->stream>>>(s, ctx->d_perm);
    } else {
        int hb = 1;
        while ((1ull << (2 * hb)) < (unsigned long long)s.Nglobal) ++hb;
        k_assign_feistel<<<(unsigned int)((s.N + 255) / 256), 256, 0, ctx->stream>>>(s, ctx->seed, ctx->round_counter, hb);
    }
    ctx->launches++;
    CK(cudaGetLastError());
    ctx->round_counter++;
    ctx->n_assigned = round + 1;
    return 0;
}

extern "C" int hmy_queue_perm(hmy_ctx* ctx, const int64_t* perm_host) {
    CK(cudaSetDevice(ctx->device));
    if (!ctx->have_data || !ctx->have_params) FAIL("hmy_queue_perm: set params and data first");
    if (!use_tc5(ctx)) FAIL("hmy_queue_perm: this context does not run one round ahead (counter \"lookahead\" is 0): pass the permutation to hmy_kmeans_round");
    if (ctx->n_assigned > ctx->n_done + (ctx->have_init ? 1 : 0)) FAIL("hmy_queue_perm: the next round already has its permutation");
    return assign_round(ctx, perm_host, ctx->n_assigned);
}

static int launch_tc5(hmy_ctx* ctx, int mode) {
    HmyDev s = ctx->st;
    const long long r = ctx->n_done;
    s.Told = ctx->t5_told[ctx->told_cur]; s.Told_next = ctx->t5_told[ctx->told_cur ^ 1];
    s.Rsum = ctx->t5_rsum[ctx->rsum_cur]; s.Rsum_next = ctx->t5_rsum[ctx->rsum_cur ^ 1];
    s.Dnew = ctx->t5_dnew;
    s.write_R = ctx->write_r;
    {   // every stage leaves its objective sums in its own ring slot: rounds can be launched back to back and read later
        const int slot = (int)(ctx->stages_launched % 16);
        s.obj = ctx->objring + 4 * slot; s.obj_out = ctx->objring + 64 + 2 * slot;
        CK(cudaMemsetAsync(s.obj, 0, 4 * sizeof(double), ctx->stream));
        CK(cudaMemsetAsync(s.Yacc, 0, (size_t)s.K * s.dp * sizeof(double), ctx->stream));
    }
    if (mode == 1) { s.blk_next = ctx->blkbuf[0]; s.Told = nullptr; s.Told_next = ctx->t5_told[ctx->told_cur]; }
    else { s.blk = ctx->blkbuf[r & 1]; s.blk_next = ctx->blkbuf[(r + 1) & 1]; }
    unsigned long long base = ctx->bar_count64;
    void* args[] = {&s, &mode, &base};
    if (ctx->fused) s.x5_seq = ++ctx->x5_seq;
    if (launch(ctx, ctx->fused ? ctx->fn_tc5_multi : ctx->fn_tc5, dim3(ctx->G_tc5), dim3(T5_THREADS), args, ctx->smem_tc5, true)) return 1;
    ctx->bar_count64 += (unsigned long long)ctx->G_tc5 * (unsigned long long)(mode == 1 ? 1 : s.nblk);
    ctx->r_valid = ctx->write_r != 0;
    ctx->t5_state = true;
    ctx->stages_launched++;
    return 0;
}

// objective sums of the last n tc5 stages (oldest first): each stage left them in its ring slot
static int fetch_obj_tc5_n(hmy_ctx* ctx, int n, double* out3n) {
    if (n < 1 || n > 16 || n > ctx->stages_launched) FAIL("hmy_objectives: n must be in 1..16 and at most the number of stages run");
    double h[16 * 6];
    CK(cudaMemcpyAsync(h, ctx->objring, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < n; ++i) {
        const int slot = (int)((ctx->stages_launched - n + i) % 16);
        const double* o = h + 4 * slot;
        if (ctx->fused) {
            // sums over all ranks (rank order) and the cross-entropy term in 2^-30 fixed point: identical on every rank
            long long fx; std::memcpy(&fx, &o[3], sizeof fx);
            out3n[3 * i] = h[64 + 2 * slot]; out3n[3 * i + 1] = h[64 + 2 * slot + 1]; out3n[3 * i + 2] = (double)fx / 1073741824.0;
        } else { out3n[3 * i] = o[0]; out3n[3 * i + 1] = o[1]; out3n[3 * i + 2] = o[2]; }
    }
    return 0;
}
static int fetch_obj_tc5(hmy_ctx* ctx, double obj[3]) {
    double o[3];
    if (fetch_obj_tc5_n(ctx, 1, o)) return 1;
    if (obj) { obj[0] = o[0]; obj[1] = o[1]; obj[2] = o[2]; }
    return 0;
}

extern "C" int hmy_objectives(hmy_ctx* ctx, int n, double* obj_3n) {
    CK(cudaSetDevice(ctx->device));
    if (!obj_3n) FAIL("hmy_objectives: NULL output");
    if (!use_tc5(ctx) || !ctx->t5_state) FAIL("hmy_objectives: only contexts with counter \"lookahead\" = 1 keep the objective sums of past rounds");
    return fetch_obj_tc5_n(ctx, n, obj_3n);
}

// ---- a2: init ------------------------------------------------------------------------------
extern "C" int hmy_init_from_centroids(hmy_ctx* ctx, const float* Y0, double obj[3]) {
    HmyDev& st = ctx->st;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->have_data || !ctx->have_params) FAIL("hmy_init_from_centroids: set params and data first");
    // unit-length centroids (harmony.py:377), K x dp zero padded
    std::vector<float> Y((size_t)st.K * st.dp, 0.f);
    for (int k = 0; k < st.K; ++k) {
        double ss = 0.0;
        for (int j = 0; j < st.d; ++j) ss += (double)Y0[(size_t)k * st.d + j] * Y0[(size_t)k * st.d + j];
        const double inv = 1.0 / std::sqrt(ss);
        for (int j = 0; j < st.d; ++j) Y[(size_t)k * st.dp + j] = (float)(Y0[(size_t)k * st.d + j] * inv);
    }
    CK(cudaMemcpyAsync(st.Yhat, Y.data(), Y.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));          // Y is a stack-lifetime host buffer
    if (use_tc5(ctx)) {
        // the init assignment also accumulates the sums the FIRST round's blocks remove: it needs that round's blocks
        if (st.ncombo >= (1 << 23)) FAIL("too many covariate combinations for the annotated block lists (>= 2^23)");
        ctx->n_done = 0;
        if (ctx->n_assigned == 0) { if (assign_round(ctx, nullptr, 0)) return 1; }     // device permutation
        else if (ctx->n_assigned != 1) FAIL("hmy_init_from_centroids: more than one permutation queued");
        CK(cudaMemsetAsync(ctx->t5_dnew, 0, ctx->t5_table_floats * sizeof(float), ctx->stream));
        CK(cudaMemsetAsync(ctx->t5_told[ctx->told_cur], 0, ctx->t5_table_floats * sizeof(float), ctx->stream));
        if (timer_begin(ctx, ctx->ev_init)) return 1;
        if (launch_tc5(ctx, 1)) return 1;
        if (timer_end(ctx, ctx->ev_init)) return 1;
        ctx->rsum_cur ^= 1;
        swap_centroids(ctx);
        ctx->have_init = true;
        return fetch_obj_tc5(ctx, obj);
    }
    if (!ctx->legacy_ok) FAIL("this (K, B, d, block_size) needs the tensor-memory round kernel (K <= 128, d <= 64, <= 32 blocks; single GPU or "
                              "fused exchange): the other round kernels keep K x B tables in shared memory and do not fit");
    ctx->t5_state = false; ctx->r_valid = true;
    CK(cudaMemsetAsync(ctx->zero_round, 0, ctx->zero_round_bytes, ctx->stream));     // obj | Ofresh | Yacc | Told | Dnew
    if (timer_begin(ctx, ctx->ev_init)) return 1;
    if (ctx->persistent && (!ctx->ar || ctx->fused)) {
        st.xseq_base = ctx->xseq;
        if (ctx->fused) ctx->xseq += 1;
        HmyDev s = st; int mode = 1; unsigned int gen = ctx->gen;
        void* args[] = {&s, &mode, &gen};
        if (launch_persistent(ctx, args)) return 1;
        ctx->gen += 1;
    } else {
        if (staged_round(ctx, 2, 0)) return 1;
        if (allreduce(ctx, st.obj, 4 + (int64_t)st.B * st.K, 1)) return 1;     // objective sums | Ofresh
        if (allreduce(ctx, st.Yacc, (int64_t)st.K * st.dp, 1)) return 1;
        if (staged_tables(ctx, 2, 1)) return 1;
    }
    if (timer_end(ctx, ctx->ev_init)) return 1;
    swap_centroids(ctx);
    ctx->have_init = true;
    return fetch_obj(ctx, obj);
}

// ---- optional: k-means++ / Lloyd initialisation on the device (hmy_kmeans_init.cuh) -----------

// Per-rank record of the exchange that precedes the first collective of a sharded initialisation:
// ok, K, d, n_global, cell_offset, n_local, max_iter, tol, seed >> 32, seed & 0xFFFFFFFF (all exact in fp64).
#define HMY_KMI_AGREE 10

static int record_rank(hmy_ctx* ctx, int rank, int world) {
    if (world > ctx->kmi_agree_world) {
        if (dev_alloc(ctx, &ctx->kmi_agree, (size_t)world * HMY_KMI_AGREE)) return 1;
        ctx->kmi_agree_world = world;
    }
    ctx->rank = rank; ctx->world = world;
    return 0;
}

// Cells sharded over ranks (n_local < n_global).  Every collective below is entered by every rank the same number of
// times: the only decisions between them are taken from all-reduced data (identical on every rank) or from checks whose
// inputs are identical on every rank.  A rank that stopped alone would leave the others waiting in a collective.
static int kmeans_init_sharded(hmy_ctx* ctx, uint64_t seed, int max_iter, double tol, float* Y_host, double info[3]) {
    HmyDev& st = ctx->st;
    if (!ctx->ar) FAIL("hmy_kmeans_init: the context holds a shard of the cells (n_local < n_global) and needs the sum "
                       "all-reduce over ranks: call hmy_set_allreduce first");
    if (ctx->rank < 0) FAIL("hmy_kmeans_init: the context holds a shard of the cells (n_local < n_global) and needs its "
                            "rank: call hmy_set_rank (or hmy_comm_attach) first");
    // checks that depend on the global shape only: the same outcome on every rank, so they may fail before any collective
    const int K = st.K, dp = st.dp, S = 2 + dp, W = ctx->world, R = ctx->rank;
    if (st.Nglobal < K) FAIL("hmy_kmeans_init: fewer cells than clusters");
    if (st.Nglobal > (1LL << 32)) FAIL("hmy_kmeans_init: sharded initialisation supports at most 2^32 cells");
    const size_t smem_lloyd = ((size_t)K * (dp | 1) + K + (size_t)K * dp + (size_t)(HMY_KMI_THREADS / 32) * dp) * sizeof(float) + (size_t)K * sizeof(unsigned int);
    if (smem_lloyd > 200 * 1024) FAIL("hmy_kmeans_init: K * d too large for the shared-memory Lloyd kernel (K (2 d + 2) floats <= 200 KB)");
    const size_t nS = (size_t)K * dp, nT = nS + K + 1;            // Lloyd table [sums K dp | counts K | inertia]
    // checks and allocations of this rank: their outcome is exchanged before the first collective that depends on them
    std::string local_err;
    if (!ctx->have_data) local_err = "hmy_kmeans_init: upload the data first";
    else if (!Y_host) local_err = "hmy_kmeans_init: NULL output";
    else if (max_iter < 0 || !(tol >= 0.0)) local_err = "hmy_kmeans_init: max_iter and tol must be non-negative";
    float *mind2 = nullptr, *C = nullptr; unsigned long long* best = nullptr; unsigned int* counts = nullptr;
    double *slots = nullptr, *tab = nullptr, *scal = nullptr; int* fail = nullptr;
    std::vector<void*> tmp;
    auto cleanup = [&]() { for (void* p : tmp) cudaFree(p); };
    auto dev = [&](void** p, size_t bytes) {
        if (!local_err.empty()) return;
        const cudaError_t e = cudaMalloc(p, bytes);
        if (e == cudaSuccess) { tmp.push_back(*p); return; }
        cudaGetLastError();
        local_err = std::string("hmy_kmeans_init: cudaMalloc failed: ") + cudaGetErrorString(e);
    };
    dev((void**)&mind2, (size_t)st.N * sizeof(float));
    dev((void**)&C, nS * sizeof(float));
    dev((void**)&best, (size_t)K * sizeof(unsigned long long));
    dev((void**)&counts, (size_t)K * sizeof(unsigned int));
    dev((void**)&slots, (size_t)W * S * sizeof(double));
    dev((void**)&tab, nT * sizeof(double));
    dev((void**)&scal, 4 * sizeof(double));
    dev((void**)&fail, sizeof(int));
    if (local_err.empty()) {
        const cudaError_t e = cudaFuncSetAttribute((const void*)k_lloyd_assign, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_lloyd);
        if (e != cudaSuccess) { cudaGetLastError(); local_err = std::string("hmy_kmeans_init: ") + cudaGetErrorString(e); }
    }
#define KCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); char b_[512]; snprintf(b_, sizeof b_, "hmy_kmeans_init: %s failed: %s", #call, cudaGetErrorString(e_)); ctx->err = b_; return 1; } } while (0)
#define KAR(p, n) do { if (allreduce(ctx, (p), (int64_t)(n), 1)) { cleanup(); return 1; } } while (0)
    // every rank's checks, arguments and cell range, gathered exactly (one slot per rank, zeros elsewhere)
    {
        std::vector<double> ag((size_t)W * HMY_KMI_AGREE, 0.0);
        double* a = ag.data() + (size_t)R * HMY_KMI_AGREE;
        const double mine[HMY_KMI_AGREE] = {local_err.empty() ? 1.0 : 0.0, (double)K, (double)st.d, (double)st.Nglobal,
                                            (double)st.cell_offset, (double)st.N, (double)max_iter, tol >= 0.0 ? tol : -1.0,
                                            (double)(seed >> 32), (double)(seed & 0xFFFFFFFFull)};
        std::copy(mine, mine + HMY_KMI_AGREE, a);
        KCK(cudaMemcpyAsync(ctx->kmi_agree, ag.data(), ag.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        KAR(ctx->kmi_agree, ag.size());
        KCK(cudaMemcpyAsync(ag.data(), ctx->kmi_agree, ag.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        KCK(cudaStreamSynchronize(ctx->stream));
        if (!local_err.empty()) { cleanup(); FAIL(local_err); }
        std::vector<std::pair<double, double>> ranges;
        for (int r = 0; r < W; ++r) {
            const double* o = ag.data() + (size_t)r * HMY_KMI_AGREE;
            if (o[0] != 1.0) { cleanup(); ctx->err = "hmy_kmeans_init: rank " + std::to_string(r) + " failed its checks (see its error)"; return 1; }
            for (int i = 1; i < HMY_KMI_AGREE; ++i)
                if (i != 4 && i != 5 && o[i] != mine[i]) {
                    cleanup(); FAIL("hmy_kmeans_init: the ranks disagree on K, d, n_global, seed, max_iter or tol");
                }
            ranges.emplace_back(o[4], o[5]);
        }
        std::sort(ranges.begin(), ranges.end());
        double next = 0.0;
        for (auto& rg : ranges) { if (rg.first != next) break; next += rg.second; }
        if (next != (double)st.Nglobal) { cleanup(); FAIL("hmy_kmeans_init: the ranks' cell ranges do not cover the n_global cells exactly once"); }
    }
    // seeding: one slot exchange per centre, no host synchronisation until the end
    KCK(cudaMemsetAsync(best, 0xFF, (size_t)K * sizeof(unsigned long long), ctx->stream));
    KCK(cudaMemsetAsync(C, 0, nS * sizeof(float), ctx->stream));
    KCK(cudaMemsetAsync(fail, 0, sizeof(int), ctx->stream));
    const long long first_id = (long long)(hmy_splitmix64((unsigned long long)seed) % (unsigned long long)st.Nglobal);
    const unsigned int grid = (unsigned int)std::min<long long>(4LL * ctx->sms, (st.N + (HMY_KMI_THREADS / 32) - 1) / (HMY_KMI_THREADS / 32));
    for (int c = 0; c < K; ++c) {
        if (c > 0) {
            k_kmpp_pass_sharded<<<grid, HMY_KMI_THREADS, dp * sizeof(float), ctx->stream>>>(st, C, c, (unsigned long long)seed, mind2, best);
            ctx->launches++;
        }
        k_kmpp_publish<<<1, 256, 0, ctx->stream>>>(st, best, c, first_id, R, W, slots);
        KCK(cudaGetLastError());
        KAR(slots, (size_t)W * S);
        k_kmpp_pick<<<1, 64, 0, ctx->stream>>>(slots, W, dp, c, C, fail);
        ctx->launches += 2;
    }
    KCK(cudaGetLastError());
    {
        int hfail = 0;
        KCK(cudaMemcpyAsync(&hfail, fail, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        KCK(cudaStreamSynchronize(ctx->stream));
        if (hfail) { cleanup(); FAIL("hmy_kmeans_init: fewer distinct cells than clusters"); }   // the same on every rank
    }
    // Lloyd: one all-reduce of the table, one of the "another iteration" votes; the loop runs while any rank votes for it
    double h[4] = {0.0, 0.0, 0.0, 0.0};   // squared shift | mean feature variance | votes | inertia
    int iters = 0;
    for (int it = 0; it < max_iter; ++it) {
        KCK(cudaMemsetAsync(tab, 0, nT * sizeof(double), ctx->stream));
        KCK(cudaMemsetAsync(counts, 0, (size_t)K * sizeof(unsigned int), ctx->stream));
        k_lloyd_assign<<<grid, HMY_KMI_THREADS, smem_lloyd, ctx->stream>>>(st, C, tab, counts, tab + nS + K);
        k_lloyd_pack_counts<<<1, 256, 0, ctx->stream>>>(counts, K, tab + nS);
        KCK(cudaGetLastError());
        KAR(tab, nT);
        k_lloyd_update_global<<<1, 256, 0, ctx->stream>>>(st, C, tab, tol, scal);
        KCK(cudaGetLastError());
        KAR(scal + 2, 1);
        ctx->launches += 3;
        KCK(cudaMemcpyAsync(h, scal, 4 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        KCK(cudaStreamSynchronize(ctx->stream));
        iters = it + 1;
        if (h[2] == 0.0) break;
    }
    // rank 0's centres and info to everyone
    {
        const double tail[3] = {(double)iters, h[3], h[0]};
        const double none[3] = {0.0, 0.0, 0.0};
        k_kmi_share<<<(unsigned int)((nS + 255) / 256), 256, 0, ctx->stream>>>(C, nS, R == 0, tab);
        ctx->launches++;
        KCK(cudaGetLastError());
        KCK(cudaMemcpyAsync(tab + nS, R == 0 ? tail : none, 3 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        KAR(tab, nS + 3);
        std::vector<double> out(nS + 3);
        KCK(cudaMemcpyAsync(out.data(), tab, out.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        KCK(cudaStreamSynchronize(ctx->stream));
        for (int k = 0; k < K; ++k) for (int j = 0; j < st.d; ++j) Y_host[(size_t)k * st.d + j] = (float)out[(size_t)k * dp + j];
        if (info) { info[0] = out[nS]; info[1] = out[nS + 1]; info[2] = out[nS + 2]; }
    }
    cleanup();
#undef KAR
#undef KCK
    return 0;
}

extern "C" int hmy_kmeans_init(hmy_ctx* ctx, uint64_t seed, int max_iter, double tol, float* Y_host, double info[3]) {
    HmyDev& st = ctx->st;
    CK(cudaSetDevice(ctx->device));
    if (st.N < st.Nglobal) return kmeans_init_sharded(ctx, seed, max_iter, tol, Y_host, info);
    if (!ctx->have_data) FAIL("hmy_kmeans_init: upload the data first");
    if (!Y_host) FAIL("hmy_kmeans_init: NULL output");
    if (max_iter < 0 || !(tol >= 0.0)) FAIL("hmy_kmeans_init: max_iter and tol must be non-negative");
    if (st.N < st.K) FAIL("hmy_kmeans_init: fewer cells than clusters");
    const int K = st.K, dp = st.dp;
    const size_t smem_lloyd = ((size_t)K * (dp | 1) + K + (size_t)K * dp + (size_t)(HMY_KMI_THREADS / 32) * dp) * sizeof(float) + (size_t)K * sizeof(unsigned int);
    if (smem_lloyd > 200 * 1024) FAIL("hmy_kmeans_init: K * d too large for the shared-memory Lloyd kernel (K (2 d + 2) floats <= 200 KB)");
    CK(cudaFuncSetAttribute((const void*)k_lloyd_assign, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_lloyd));
    float *mind2 = nullptr, *C = nullptr; unsigned long long* best = nullptr; double *sums = nullptr, *scal = nullptr; unsigned int* counts = nullptr;
    std::vector<void*> tmp;
    auto cleanup = [&]() { for (void* p : tmp) cudaFree(p); };
#define KCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); char b_[512]; snprintf(b_, sizeof b_, "hmy_kmeans_init: %s failed: %s", #call, cudaGetErrorString(e_)); ctx->err = b_; return 1; } } while (0)
    KCK(cudaMalloc((void**)&mind2, (size_t)st.N * sizeof(float))); tmp.push_back(mind2);
    KCK(cudaMalloc((void**)&C, (size_t)K * dp * sizeof(float))); tmp.push_back(C);
    KCK(cudaMalloc((void**)&best, (size_t)K * sizeof(unsigned long long))); tmp.push_back(best);
    KCK(cudaMalloc((void**)&sums, (size_t)K * dp * sizeof(double))); tmp.push_back(sums);
    KCK(cudaMalloc((void**)&counts, (size_t)K * sizeof(unsigned int))); tmp.push_back(counts);
    KCK(cudaMalloc((void**)&scal, 4 * sizeof(double))); tmp.push_back(scal);
    KCK(cudaMemsetAsync(best, 0xFF, (size_t)K * sizeof(unsigned long long), ctx->stream));
    KCK(cudaMemsetAsync(C, 0, (size_t)K * dp * sizeof(float), ctx->stream));
    // centre 0: uniform over the cells (by caller index, so the draw does not depend on the storage order)
    const long long first_id = (long long)(hmy_splitmix64((unsigned long long)seed) % (unsigned long long)st.Nglobal);
    int first_pos_i = 0;
    KCK(cudaMemcpyAsync(&first_pos_i, st.pos_of + (first_id - st.cell_offset), sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    KCK(cudaStreamSynchronize(ctx->stream));
    const long long first_pos = first_pos_i;
    const unsigned int grid = (unsigned int)std::min<long long>(4LL * ctx->sms, (st.N + (HMY_KMI_THREADS / 32) - 1) / (HMY_KMI_THREADS / 32));
    for (int c = 1; c < K; ++c) {
        k_kmpp_pass<<<grid, HMY_KMI_THREADS, dp * sizeof(float), ctx->stream>>>(st, best, first_pos, c, (unsigned long long)seed, mind2, best);
        ctx->launches++;
    }
    KCK(cudaGetLastError());
    {
        std::vector<unsigned long long> hb(K);
        KCK(cudaMemcpyAsync(hb.data(), best, (size_t)K * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
        KCK(cudaStreamSynchronize(ctx->stream));
        for (int c = 1; c < K; ++c)
            if (hb[c] == ~0ull) { cleanup(); FAIL("hmy_kmeans_init: fewer distinct cells than clusters"); }
    }
    k_kmpp_gather<<<K, 64, 0, ctx->stream>>>(st, best, first_pos, C);
    ctx->launches++;
    KCK(cudaGetLastError());
    double h[3] = {0.0, 0.0, 0.0};       // inertia | squared shift | mean feature variance
    int iters = 0;
    for (int it = 0; it < max_iter; ++it) {
        KCK(cudaMemsetAsync(sums, 0, (size_t)K * dp * sizeof(double), ctx->stream));
        KCK(cudaMemsetAsync(counts, 0, (size_t)K * sizeof(unsigned int), ctx->stream));
        KCK(cudaMemsetAsync(scal, 0, 4 * sizeof(double), ctx->stream));
        k_lloyd_assign<<<grid, HMY_KMI_THREADS, smem_lloyd, ctx->stream>>>(st, C, sums, counts, scal);
        k_lloyd_update<<<1, 256, 0, ctx->stream>>>(st, C, sums, counts, scal + 1);
        ctx->launches += 2;
        KCK(cudaGetLastError());
        KCK(cudaMemcpyAsync(h, scal, 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        KCK(cudaStreamSynchronize(ctx->stream));
        iters = it + 1;
        if (h[1] <= tol * h[2]) break;                          // sklearn: centre shift^2 <= tol * mean(var(X, axis=0))
    }
    std::vector<float> Yp((size_t)K * dp);
    KCK(cudaMemcpyAsync(Yp.data(), C, Yp.size() * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    KCK(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < K; ++k) for (int j = 0; j < st.d; ++j) Y_host[(size_t)k * st.d + j] = Yp[(size_t)k * dp + j];
    if (info) { info[0] = (double)iters; info[1] = h[0]; info[2] = h[1]; }
    cleanup();
#undef KCK
    return 0;
}

// ---- a3/a4/a5: one k-means round -----------------------------------------------------------
extern "C" int hmy_kmeans_round(hmy_ctx* ctx, const int64_t* perm_host, double obj[3]) {
    HmyDev& st = ctx->st;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->have_init) FAIL("hmy_kmeans_round: call hmy_init_from_centroids first");
    if (use_tc5(ctx)) {
        // one round ahead: perm_host (or the device permutation) is the NEXT round's; this round's was queued by the
        // previous call (the first one by hmy_queue_perm / hmy_init_from_centroids)
        if (!ctx->t5_state) FAIL("hmy_kmeans_round: the context switched kernels after init");
        const long long r = ctx->n_done;
        if (ctx->n_assigned == r + 1) { if (assign_round(ctx, perm_host, r + 1)) return 1; }
        else if (ctx->n_assigned != r + 2 || perm_host) FAIL("hmy_kmeans_round: permutation queue out of step");
        {
            HmyDev s = st;
            s.blk = ctx->blkbuf[r & 1]; s.blk_next = ctx->blkbuf[(r + 1) & 1];
            const size_t sm = ((size_t)st.nblk * HMY_LIST_THREADS + st.nblk) * sizeof(unsigned int);
            HmyDev c1 = s; c1.list2 = nullptr;
            k_block_lists<<<ctx->list_chunks, HMY_LIST_THREADS, sm, ctx->stream>>>(c1, ctx->d_cnt, 1);
            k_block_scan<<<1, 32 * std::min(32, st.nblk), 0, ctx->stream>>>(s, ctx->d_cnt, ctx->list_chunks);
            k_block_lists<<<ctx->list_chunks, HMY_LIST_THREADS, sm, ctx->stream>>>(s, ctx->d_cnt, 0);
            ctx->launches += 3;
            CK(cudaGetLastError());
        }
        CK(cudaMemsetAsync(ctx->t5_dnew, 0, ctx->t5_table_floats * sizeof(float), ctx->stream));
        CK(cudaMemsetAsync(ctx->t5_told[ctx->told_cur ^ 1], 0, ctx->t5_table_floats * sizeof(float), ctx->stream));
        if (timer_begin(ctx, ctx->ev_round)) return 1;
        if (launch_tc5(ctx, 0)) return 1;
        if (timer_end(ctx, ctx->ev_round)) return 1;
        ctx->told_cur ^= 1; ctx->rsum_cur ^= 1;
        ctx->n_done++;
        swap_centroids(ctx);
        ctx->rounds++;
        if (!obj) return 0;                  // the caller reads the sums later (hmy_objectives): no host round trip now
        return fetch_obj_tc5(ctx, obj);
    }
    // block of every cell for this round (harmony.py:471-475)
    if (perm_host) {
        if (!ctx->d_perm) CK(cudaMalloc((void**)&ctx->d_perm, (size_t)st.Nglobal * sizeof(long long)));
        CK(cudaMemcpyAsync(ctx->d_perm, perm_host, (size_t)st.Nglobal * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
        k_assign_from_perm<<<(unsigned int)((st.Nglobal + 255) / 256), 256, 0, ctx->stream>>>(st, ctx->d_perm);
    } else {
        int hb = 1;
        while ((1ull << (2 * hb)) < (unsigned long long)st.Nglobal) ++hb;
        k_assign_feistel<<<(unsigned int)((st.N + 255) / 256), 256, 0, ctx->stream>>>(st, ctx->seed, ctx->round_counter, hb);
    }
    ctx->launches++;
    CK(cudaGetLastError());
    ctx->round_counter++;
    {   // per-block cell lists (stable counting sort over position chunks)
        const size_t sm = ((size_t)st.nblk * HMY_LIST_THREADS + st.nblk) * sizeof(unsigned int);
        HmyDev sl = st; sl.list2 = nullptr;            // plain position lists (the annotated ones belong to the tc5 path)
        k_block_lists<<<ctx->list_chunks, HMY_LIST_THREADS, sm, ctx->stream>>>(sl, ctx->d_cnt, 1);
        k_block_scan<<<1, 32 * std::min(32, st.nblk), 0, ctx->stream>>>(sl, ctx->d_cnt, ctx->list_chunks);
        k_block_lists<<<ctx->list_chunks, HMY_LIST_THREADS, sm, ctx->stream>>>(sl, ctx->d_cnt, 0);
        ctx->launches += 3;
        CK(cudaGetLastError());
    }
    CK(cudaMemsetAsync(ctx->zero_round, 0, ctx->zero_round_bytes, ctx->stream));     // obj | Ofresh | Yacc | Told | Dnew
    if (timer_begin(ctx, ctx->ev_round)) return 1;
    if (ctx->persistent && (!ctx->ar || ctx->fused)) {
        st.xseq_base = ctx->xseq;
        if (ctx->fused) ctx->xseq += st.xrelaxed ? 1u : (unsigned int)st.nblk + 1u;
        HmyDev s = st; int mode = 0; unsigned int gen = ctx->gen;
        void* args[] = {&s, &mode, &gen};
        if (launch_persistent(ctx, args)) return 1;
        ctx->gen += (unsigned int)st.nblk + 1u;
    } else {
        const int64_t nT = (int64_t)st.nblk * st.B * st.K, BK = (int64_t)st.B * st.K;
        if (staged_round(ctx, 0, 0)) return 1;
        if (allreduce(ctx, st.Told, nT, 0)) return 1;
        if (staged_tables(ctx, 0, 0)) return 1;
        for (int blk = 0; blk < st.nblk; ++blk) {
            if (staged_round(ctx, 1, blk)) return 1;
            if (allreduce(ctx, st.Dnew + (size_t)blk * BK, BK, 0)) return 1;
            if (blk + 1 < st.nblk && staged_tables(ctx, 1, blk + 1)) return 1;
        }
        if (allreduce(ctx, st.Yacc, (int64_t)st.K * st.dp, 1)) return 1;
        if (allreduce(ctx, st.obj, 4 + (int64_t)st.B * st.K, 1)) return 1;     // objective sums | Ofresh
        if (staged_tables(ctx, 2, 0)) return 1;
    }
    if (timer_end(ctx, ctx->ev_round)) return 1;
    swap_centroids(ctx);
    ctx->rounds++;
    return fetch_obj(ctx, obj);
}

// ---- a7: ridge correction -------------------------------------------------------------------
extern "C" int hmy_ridge_correct(hmy_ctx* ctx) {
    HmyDev& st = ctx->st;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->have_init) FAIL("hmy_ridge_correct: call hmy_init_from_centroids first");
    if (!ctx->r_valid) FAIL("hmy_ridge_correct: the last stage did not store R (option write_r = 0)");
    CK(cudaMemsetAsync(ctx->zero_ridge, 0, ctx->zero_ridge_bytes, ctx->stream));
    CK(cudaMemsetAsync(st.Yacc, 0, (size_t)st.K * st.dp * sizeof(double), ctx->stream));
    if (timer_begin(ctx, ctx->ev_ridge)) return 1;
    const int grid_m = std::min(ctx->grid_mom, std::max(1, st.nseg));
    const int grid_a = std::min(ctx->grid_ridge, std::max(1, st.nseg));
    CK(cudaMemsetAsync(st.wmax, 0, sizeof(float), ctx->stream));
    {
        HmyDev s = st; float zs = ctx->zscale; void* args[] = {&s, &zs};
        if (launch(ctx, ctx->fn_mom, dim3(grid_m), dim3(ctx->ridge_threads), args, ctx->smem_mom, false)) return 1;
    }
    {
        const int64_t nG = (int64_t)st.K * (st.B + 1) * (st.B + 1), nM = (int64_t)(st.B + 1) * st.K * st.dp;
        if (allreduce(ctx, st.Gram, nG + nM, 1)) return 1;
    }
    {
        HmyDev s = st; void* args[] = {&s};
        if (launch(ctx, (const void*)k_ridge_solve, dim3(st.K), dim3(128), args, ctx->smem_solve, false)) return 1;
    }
    {
        HmyDev s = st; const float* wm = st.wmax; void* args[] = {&s, &wm};
        if (launch(ctx, ctx->fn_apply, dim3(grid_a), dim3(ctx->ridge_threads), args, ctx->smem_apply, false)) return 1;
    }
    if (allreduce(ctx, st.Yacc, (int64_t)st.K * st.dp, 1)) return 1;
    {
        // centroids the next cluster() starts from (harmony.py:443 with the new Z_cos): they
        // replace the pending ones, not the ones the last round used
        HmyDev s = st; s.Ynext = st.Yhat;
        int what = 2, mode = 2;
        void* args[] = {&s, &what, &mode};
        if (launch(ctx, (const void*)k_tables, dim3(1), dim3(HMY_THREADS), args, 0, false)) return 1;
    }
    if (!ctx->ridge_mma && split_zcos(ctx)) return 1;   // operand rows of the round kernel follow the new Z_cos (the tensor-core apply pass writes them itself)
    if (timer_end(ctx, ctx->ev_ridge)) return 1;
    ctx->ridge_passes++;
    return 0;
}

// ---- property reads --------------------------------------------------------------------------
static int get_cells(hmy_ctx* ctx, const float* src, int sp, int w, void* host_out, int64_t bytes) {
    HmyDev& st = ctx->st;
    const size_t need = (size_t)st.N * w * sizeof(float);
    if ((size_t)bytes != need) FAIL("hmy_get: wrong buffer size");
    if (ctx->tmp_bytes < need) {
        if (ctx->d_tmp) cudaFree(ctx->d_tmp);
        ctx->d_tmp = nullptr; ctx->tmp_bytes = 0;
        CK(cudaMalloc((void**)&ctx->d_tmp, need));
        ctx->tmp_bytes = need;
    }
    const long long threads = st.N * 32;
    k_unsort_rows<<<(unsigned int)((threads + 255) / 256), 256, 0, ctx->stream>>>(src, sp, ctx->d_tmp, w, st.order, st.N);
    ctx->launches++;
    CK(cudaGetLastError());
    if (need >= (1u << 20) && host_is_pinned(host_out)) {       // page-locked destination: one DMA, no bounce, no host copy
        CK(cudaMemcpyAsync(host_out, ctx->d_tmp, need, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->dma_direct++;
        return 0;
    }
    // device -> pinned bounce buffer -> caller's (pageable, usually untouched) array, double buffered:
    // the DMA of chunk i+1 overlaps the host copy (and first-touch page faults) of chunk i
    constexpr size_t CHUNK = HMY_STAGE_CHUNK;
    if (ensure_stage(ctx)) return 1;
    const unsigned char* src8 = reinterpret_cast<const unsigned char*>(ctx->d_tmp);
    unsigned char* dst8 = reinterpret_cast<unsigned char*>(host_out);
    const size_t nchunk = (need + CHUNK - 1) / CHUNK;
    for (size_t i = 0; i <= nchunk; ++i) {
        if (i < nchunk) {
            const size_t off = i * CHUNK, len = std::min(CHUNK, need - off);
            CK(cudaMemcpyAsync(ctx->h_stage[i & 1], src8 + off, len, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaEventRecord(ctx->ev_stage[i & 1], ctx->stream));
        }
        if (i > 0) {
            const size_t j = i - 1, off = j * CHUNK, len = std::min(CHUNK, need - off);
            CK(cudaEventSynchronize(ctx->ev_stage[j & 1]));
            // the destination is usually a fresh (never touched) array: its first-touch page faults
            // dominate, so the copy is spread over a few host threads
            const unsigned char* hb = ctx->h_stage[j & 1];
            parallel_ranges((long long)len, len >= (2u << 20) ? host_threads() : 1,
                            [&](int, long long lo, long long hi) { std::memcpy(dst8 + off + lo, hb + lo, (size_t)(hi - lo)); });
        }
    }
    return 0;
}

extern "C" int hmy_get(hmy_ctx* ctx, int which, void* host_out, int64_t bytes) {
    HmyDev& st = ctx->st;
    CK(cudaSetDevice(ctx->device));
    if (!host_out) FAIL("hmy_get: NULL output");
    switch (which) {
        case HMY_Z_CORR: return get_cells(ctx, st.Zcorr, st.dp, st.d, host_out, bytes);
        case HMY_Z_COS: return get_cells(ctx, st.Zcos, st.dp, st.d, host_out, bytes);
        case HMY_Z_ORIG: return get_cells(ctx, st.Zorig, st.dp, st.d, host_out, bytes);
        case HMY_R:
            if (!ctx->r_valid) FAIL("hmy_get(R): the last stage did not store R (option write_r = 0)");
            return get_cells(ctx, st.R, st.Kp, st.K, host_out, bytes);
        case HMY_Y: {
            if ((size_t)bytes != (size_t)st.K * st.d * sizeof(float)) FAIL("hmy_get(Y): wrong buffer size");
            std::vector<float> t((size_t)st.K * st.dp);
            CK(cudaMemcpyAsync(t.data(), ctx->Ylast, t.size() * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            float* o = (float*)host_out;
            for (int k = 0; k < st.K; ++k) for (int j = 0; j < st.d; ++j) o[(size_t)k * st.d + j] = t[(size_t)k * st.dp + j];
            return 0;
        }
        case HMY_O: case HMY_E: {
            if ((size_t)bytes != (size_t)st.K * st.B * sizeof(double)) FAIL("hmy_get(O/E): wrong buffer size");
            std::vector<double> t((size_t)st.B * st.K);
            std::vector<float> pr(st.B);
            CK(cudaMemcpyAsync(t.data(), st.O, t.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaMemcpyAsync(pr.data(), st.Pr_b, st.B * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            double* o = (double*)host_out;
            for (int k = 0; k < st.K; ++k) {
                double rs = 0.0;
                for (int b = 0; b < st.lev0; ++b) rs += t[(size_t)b * st.K + k];
                for (int b = 0; b < st.B; ++b)
                    o[(size_t)k * st.B + b] = (which == HMY_O) ? t[(size_t)b * st.K + k] : rs * (double)pr[b];   // E: harmony.py:388
            }
            return 0;
        }
        case 9: {   // HMY_TRACE: uint64 [grid][HMY_TRACE_SLOTS] globaltimer stamps of the last round
            const size_t n = (size_t)((use_tc5(ctx) ? ctx->G_tc5 : ctx->G) + 1) * HMY_TRACE_SLOTS * sizeof(unsigned long long);
            if (!st.trace) FAIL("hmy_get(trace): tracing is off");
            if ((size_t)bytes != n) FAIL("hmy_get(trace): wrong buffer size");
            CK(cudaStreamSynchronize(ctx->stream));
            CK(cudaMemcpy(host_out, st.trace, n, cudaMemcpyDeviceToHost));
            return 0;
        }
        case HMY_W: {
            const size_t n = (size_t)st.B * st.K * st.d;
            if ((size_t)bytes != n * sizeof(float)) FAIL("hmy_get(W): wrong buffer size");
            std::vector<float> t((size_t)st.B * st.K * st.dp);
            CK(cudaMemcpyAsync(t.data(), st.W, t.size() * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            float* o = (float*)host_out;
            for (size_t r = 0; r < (size_t)st.B * st.K; ++r) for (int j = 0; j < st.d; ++j) o[r * st.d + j] = t[r * st.dp + j];
            return 0;
        }
    }
    FAIL("hmy_get: unknown matrix id");
}

extern "C" int hmy_synchronize(hmy_ctx* ctx) {
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int hmy_set_option(hmy_ctx* ctx, const char* name, int64_t value) {
    const std::string n(name ? name : "");
    if (n == "persistent") { ctx->persistent = value != 0; return 0; }
    if (n == "seed") {
        if (ctx->n_assigned > 0) FAIL("option seed: a permutation of the current run is already queued (set the seed before init)");
        ctx->seed = (unsigned long long)value * 0x9E3779B97F4A7C15ull + 0x243F6A8885A308D3ull; ctx->round_counter = 0; return 0;
    }
    if (n == "timing") { ctx->timing = value != 0; return 0; }
    if (n == "trace") {
        // per-CTA timeline of the persistent round kernel (debug / profiling aid)
        CK(cudaSetDevice(ctx->device));
        if (value && !ctx->st.trace) {
            if (!ctx->have_params) FAIL("trace: set params first");
            const size_t slots = (size_t)(std::max(ctx->G, ctx->G_tc5) + 1) * HMY_TRACE_SLOTS;
            if (dev_alloc(ctx, &ctx->st.trace, slots)) return 1;
            CK(cudaMemset(ctx->st.trace, 0, slots * sizeof(unsigned long long)));
        }
        return 0;
    }
    if (n == "force_fused_kernel") { ctx->force_fused_kernel = value != 0; return 0; }   // codegen A/B only
    if (n == "relaxed") {
        // fused multi-GPU mode only: 1 = the K x B table crosses GPUs once per round instead of once
        // per block (Jacobi across GPUs, Gauss-Seidel inside a GPU; north_star's single exchange)
        ctx->st.xrelaxed = value != 0; return 0;
    }
    if (n == "ridge_mma") {
        if (ctx->have_params) FAIL("option ridge_mma must be set before hmy_set_params");
        ctx->want_ridge_mma = value != 0; return 0;
    }
    if (n == "mma_wn") {
        if (ctx->have_params) FAIL("option mma_wn must be set before hmy_set_params");
        ctx->force_wn = (int)value; return 0;
    }
    if (n == "mma") {
        if (ctx->have_params) FAIL("option mma must be set before hmy_set_params");
        ctx->want_mma = value != 0; return 0;
    }
    if (n == "tc5") {
        if (ctx->have_params) FAIL("option tc5 must be set before hmy_set_params");
        ctx->want_tc5 = (int)value; return 0;
    }
    if (n == "write_r") { ctx->write_r = value != 0; return 0; }
    if (n == "dbg") { ctx->st.dbg = (int)value; return 0; }          // timing experiments (wrong results); see hmy_round_tc5.cuh
    if (n == "reset") {
        // back to the freshly-uploaded state (benchmark steps restart from here)
        CK(cudaSetDevice(ctx->device));
        if (!ctx->have_data) FAIL("reset: no data");
        const long long threads = ctx->st.N * 32;
        k_reset<<<(unsigned int)((threads + 255) / 256), 256, 0, ctx->stream>>>(ctx->st);
        ctx->launches++;
        CK(cudaGetLastError());
        if (split_zcos(ctx)) return 1;
        ctx->have_init = false;
        ctx->round_counter = 0; ctx->n_assigned = 0; ctx->n_done = 0;      // the permutation stream starts over as well
        ctx->ycur = 0; ctx->st.Yhat = ctx->Ybuf[0]; ctx->st.Ynext = ctx->Ybuf[1]; ctx->Ylast = ctx->Ybuf[0];
        return 0;
    }
    FAIL("hmy_set_option: unknown option");
}

extern "C" int64_t hmy_counter(const hmy_ctx* ctx, const char* name) {
    const std::string n(name ? name : "");
    if (n == "launches") return ctx->launches;
    if (n == "rounds") return ctx->rounds;
    if (n == "ridge_passes") return ctx->ridge_passes;
    if (n == "grid") return use_tc5(ctx) ? ctx->G_tc5 : ctx->G;
    if (n == "fused") return ctx->fused ? 1 : 0;
    if (n == "smem_round") return use_tc5(ctx) ? ctx->smem_tc5 : ctx->smem_round;
    if (n == "nblk") return ctx->st.nblk;
    if (n == "ncombo") return ctx->st.ncombo;
    if (n == "mma") return ctx->use_mma ? 1 : 0;
    if (n == "ridge_mma") return ctx->ridge_mma ? 1 : 0;
    if (n == "round_threads") return use_tc5(ctx) ? T5_THREADS : ctx->round_threads;
    if (n == "tc5") return use_tc5(ctx) ? 1 : 0;
    if (n == "dma_direct") return ctx->dma_direct;
    if (n == "lookahead") return use_tc5(ctx) ? 1 : 0;      // 1: permutations are queued one round ahead (hmy_queue_perm)
    if (n == "r_valid") return ctx->r_valid ? 1 : 0;
    return -1;
}

extern "C" double hmy_timer_ms(hmy_ctx* ctx, const char* name) {
    const std::string n(name ? name : "");
    cudaSetDevice(ctx->device);
    timer_collect(ctx->ev_round, ctx->ms_round);
    timer_collect(ctx->ev_ridge, ctx->ms_ridge);
    timer_collect(ctx->ev_init, ctx->ms_init);
    if (n == "ms_init") return ctx->ms_init;
    if (n == "ms_round") return ctx->ms_round;
    if (n == "ms_ridge") return ctx->ms_ridge;
    return -1.0;
}

extern "C" int hmy_set_allreduce(hmy_ctx* ctx, hmy_allreduce_fn fn, void* user) {
    ctx->ar = fn; ctx->ar_user = user;
    return 0;
}

extern "C" int hmy_comm_export(hmy_ctx* ctx, void* handle_out_64B) {
    HmyDev& st = ctx->st;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->have_params) FAIL("hmy_comm_export: call hmy_set_params first");
    if (!ctx->use_mma && !ctx->tc5_ok) FAIL("hmy_comm_export: the fused exchange needs a tensor-core round kernel (d <= 64)");
    if (!handle_out_64B) FAIL("hmy_comm_export: NULL handle");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    if (!ctx->xbuf) {
        size_t slot = (size_t)st.B * st.K * sizeof(float);
        slot = std::max(slot, (size_t)(4 + (size_t)st.B * st.K + (size_t)st.K * st.dp) * sizeof(double));
        slot = (slot + 255) & ~(size_t)255;
        st.xslot = slot;
        st.xll_count = st.B * st.K;
        ctx->xbytes = HMY_XPAYLOAD_OFF + 2 * (size_t)HMY_MAX_WORLD * slot
                    + 2 * (size_t)HMY_MAX_WORLD * (size_t)st.xll_count * sizeof(uint2);
        if (ctx->tc5_ok) {
            // LL regions of the tensor-memory round kernel (hmy_round_tc5.cuh): per-block sums [2][nblk][W][nD], the next
            // round's removed sums [2][W][nblk nD], centroid / objective sums as double halves [2][W][2 (K dp + 2)]
            const size_t nD = (size_t)st.B * st.K + st.K, nT = (size_t)st.nblk * nD, nY = (size_t)st.K * st.dp + 2;
            ctx->xbytes = (ctx->xbytes + 255) & ~(size_t)255;
            st.x5_off_d = ctx->xbytes; ctx->xbytes += 2 * nT * HMY_MAX_WORLD * sizeof(uint2);
            st.x5_off_t = ctx->xbytes; ctx->xbytes += 2 * (size_t)HMY_MAX_WORLD * nT * sizeof(uint2);
            st.x5_off_y = ctx->xbytes; ctx->xbytes += 2 * (size_t)HMY_MAX_WORLD * 2 * nY * sizeof(uint2);
        }
        CK(cudaMalloc((void**)&ctx->xbuf, ctx->xbytes));
        CK(cudaMemset(ctx->xbuf, 0, ctx->xbytes));
    }
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, ctx->xbuf));
    std::memcpy(handle_out_64B, &h, 64);
    return 0;
}

extern "C" int hmy_comm_attach(hmy_ctx* ctx, int rank, int world, const void* all_handles) {
    HmyDev& st = ctx->st;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->xbuf) FAIL("hmy_comm_attach: call hmy_comm_export first");
    if (world < 1 || world > HMY_MAX_WORLD || rank < 0 || rank >= world) FAIL("hmy_comm_attach: bad rank / world (<= 8 ranks)");
    for (int r = 0; r < world; ++r) {
        if (r == rank) { st.xpeer[r] = ctx->xbuf; continue; }
        cudaIpcMemHandle_t h;
        std::memcpy(&h, (const unsigned char*)all_handles + (size_t)r * 64, 64);
        void* p = nullptr;
        CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        ctx->xopened.push_back(p);
        st.xpeer[r] = (unsigned char*)p;
    }
    st.xrank = rank; st.xworld = world;
    ctx->fused = world > 1;
    return record_rank(ctx, rank, world);
}

extern "C" int hmy_set_rank(hmy_ctx* ctx, int rank, int world) {
    CK(cudaSetDevice(ctx->device));
    if (world < 1 || rank < 0 || rank >= world) FAIL("hmy_set_rank: need 0 <= rank < world");
    return record_rank(ctx, rank, world);
}
