// k-means++ / Lloyd initialisation of the centroids on the device (SURVEY.md section 8(f) rank 1): the optional
// replacement of the reference's sklearn call (harmony.py:369-373: KMeans(init="k-means++", n_init=1, max_iter=25)
// on the unit-length cells) for sizes where that call dominates the wall time.  It cannot reproduce sklearn's random
// stream, so the parity configurations keep sklearn; what it is compared with is oracle/kmeans_init_oracle.py, the
// same algorithm in NumPy with the same counter-based random numbers.
//
// Runs with the plain GPU suite (tests/test_gpu_kmeans_init.py, tests/test_gpu_dist_kmeans_init.py).
//
// Seeding (k-means++, Arthur & Vassilvitskii): centre 0 uniformly; centre c with probability proportional to the
// squared distance to the nearest centre so far.  The draw is an exponential race, argmin_i E_i / D2_i with
// E_i = -log(u(seed, c, cell id)): one min-reduction, no prefix sums, and independent of how the cells are laid out
// in memory (the engine stores them sorted by covariate combination).  Lloyd: one warp per cell, lanes over clusters,
// per-CTA shared-memory sums, fp64 global sums; stops at sklearn's criterion (squared centre shift <=
// tol * mean feature variance) or after max_iter iterations.
//
// Cells sharded over ranks: because the race keys depend on the global cell id only, every rank runs the pass over its
// own cells (k_kmpp_pass_sharded, the previous centre read from the gathered centre table) and publishes its winner as
// one slot {key, global id, row} of a world x (2 + dp) fp64 table whose other slots are zero (k_kmpp_publish); a sum
// all-reduce of that table is an exact all-gather (fp32 values and ids are exact in fp64, x + 0 = x), and
// k_kmpp_pick takes the minimum by (key, global id) -- the cell a single GPU holding every cell picks.  Lloyd keeps
// k_lloyd_assign; its local sums, counts and inertia travel as one fp64 table through one all-reduce, and
// k_lloyd_update_global divides by the global cell count.
#pragma once
#include "hmy_common.cuh"

#define HMY_KMI_THREADS 256

__host__ __device__ inline unsigned long long hmy_splitmix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    unsigned long long z = x;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
// uniform in (0, 1] from (seed, step, cell id)
__host__ __device__ inline double hmy_kmi_uniform(unsigned long long seed, int step, unsigned long long id) {
    const unsigned long long h = hmy_splitmix64(hmy_splitmix64(hmy_splitmix64(seed) + (unsigned long long)step) ^ id);
    return (double)((h >> 11) + 1ull) * (1.0 / 9007199254740992.0);
}

#ifdef HMY_NONTEMPLATE_KERNELS

// One seeding step: D2 to centre `c - 1` (row `prev_pos` of Z_cos), running minimum, race for centre c.
// best[c] must be ~0ull on entry; afterwards its low 32 bits are the winner's position.
__global__ void __launch_bounds__(HMY_KMI_THREADS) k_kmpp_pass(HmyDev st, const unsigned long long* best, long long first_pos, int c,
                                                               unsigned long long seed, float* mind2, unsigned long long* best_out) {
    extern __shared__ __align__(16) unsigned char kmi_smem[];
    float* sy = reinterpret_cast<float*>(kmi_smem);                       // [dp] the newest centre
    __shared__ unsigned long long s_best[HMY_KMI_THREADS / 32];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, dp = st.dp;
    const long long prev_pos = (c == 1) ? first_pos : (long long)(best[c - 1] & 0xFFFFFFFFull);
    if (prev_pos >= st.N) return;          // the previous step found no cell at a positive distance (host reports it)
    for (int j = tid; j < dp; j += HMY_KMI_THREADS) sy[j] = st.Zcos[(size_t)prev_pos * dp + j];
    __syncthreads();
    unsigned long long mine = ~0ull;
    const long long nw = (long long)gridDim.x * (HMY_KMI_THREADS / 32);
    for (long long pos = (long long)blockIdx.x * (HMY_KMI_THREADS / 32) + warp; pos < st.N; pos += nw) {
        const float* z = st.Zcos + (size_t)pos * dp;
        float s = 0.f;
        for (int j = lane; j < dp; j += 32) { const float u = z[j] - sy[j]; s = fmaf(u, u, s); }
        s = warp_sum(s);
        if (lane == 0) {
            const float m = (c == 1) ? s : fminf(mind2[pos], s);
            mind2[pos] = m;
            if (m > 0.f) {
                const unsigned long long id = (unsigned long long)(st.cell_offset + st.order[pos]);
                const float key = (float)(-log(hmy_kmi_uniform(seed, c, id)) / (double)m);
                const unsigned long long packed = ((unsigned long long)__float_as_uint(key) << 32) | (unsigned long long)(unsigned int)pos;
                mine = packed < mine ? packed : mine;
            }
        }
    }
    if (lane == 0) s_best[warp] = mine;
    __syncthreads();
    if (tid == 0) {
        unsigned long long b = s_best[0];
        for (int w = 1; w < HMY_KMI_THREADS / 32; ++w) b = s_best[w] < b ? s_best[w] : b;
        if (b != ~0ull) atomicMin(&best_out[c], b);
    }
}

// rows of the chosen cells -> C [K][dp]
__global__ void k_kmpp_gather(HmyDev st, const unsigned long long* best, long long first_pos, float* C) {
    const int k = blockIdx.x;
    const long long pos = (k == 0) ? first_pos : (long long)(best[k] & 0xFFFFFFFFull);
    if (pos >= st.N) return;
    for (int j = threadIdx.x; j < st.dp; j += blockDim.x) C[(size_t)k * st.dp + j] = st.Zcos[(size_t)pos * st.dp + j];
}

// One Lloyd assignment pass.  sums [K][dp] fp64, counts [K], inertia [1] must be zero on entry.
__global__ void __launch_bounds__(HMY_KMI_THREADS) k_lloyd_assign(HmyDev st, const float* __restrict__ C, double* sums, unsigned int* counts, double* inertia) {
    extern __shared__ __align__(16) unsigned char kmi_smem[];
    const int K = st.K, dp = st.dp, dps = dp | 1;
    float* sC = reinterpret_cast<float*>(kmi_smem);                       // [K][dps]
    float* sN = sC + (size_t)K * dps;                                     // [K] squared norms
    float* sSum = sN + K;                                                 // [K][dp]
    float* sZ = sSum + (size_t)K * dp;                                    // [warps][dp]
    unsigned int* sCnt = reinterpret_cast<unsigned int*>(sZ + (HMY_KMI_THREADS / 32) * dp);   // [K]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int i = tid; i < K * dp; i += HMY_KMI_THREADS) { const int k = i / dp, j = i - k * dp; sC[k * dps + j] = C[i]; sSum[i] = 0.f; }
    for (int k = tid; k < K; k += HMY_KMI_THREADS) sCnt[k] = 0u;
    __syncthreads();
    for (int k = tid; k < K; k += HMY_KMI_THREADS) { float s = 0.f; for (int j = 0; j < dp; ++j) s = fmaf(sC[k * dps + j], sC[k * dps + j], s); sN[k] = s; }
    __syncthreads();
    float* mz = sZ + warp * dp;
    double my_inertia = 0.0;
    const long long nw = (long long)gridDim.x * (HMY_KMI_THREADS / 32);
    for (long long pos = (long long)blockIdx.x * (HMY_KMI_THREADS / 32) + warp; pos < st.N; pos += nw) {
        const float* z = st.Zcos + (size_t)pos * dp;
        float zn = 0.f;
        for (int j = lane; j < dp; j += 32) { const float v = z[j]; mz[j] = v; zn = fmaf(v, v, zn); }
        zn = warp_sum(zn);
        __syncwarp();
        float bestv = INFINITY; int bestk = 0x7fffffff;
        for (int k = lane; k < K; k += 32) {
            const float* ck = sC + k * dps;
            float dot = 0.f;
            for (int j = 0; j < dp; ++j) dot = fmaf(mz[j], ck[j], dot);
            const float v = sN[k] - 2.f * dot;                            // ||z - c||^2 - ||z||^2
            if (v < bestv) { bestv = v; bestk = k; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bestv, o);
            const int ok = __shfl_xor_sync(0xffffffffu, bestk, o);
            if (ov < bestv || (ov == bestv && ok < bestk)) { bestv = ov; bestk = ok; }
        }
        for (int j = lane; j < dp; j += 32) atomicAdd(&sSum[bestk * dp + j], mz[j]);
        if (lane == 0) { atomicAdd(&sCnt[bestk], 1u); my_inertia += (double)(bestv + zn); }
        __syncwarp();
    }
    __syncthreads();
    for (int i = tid; i < K * dp; i += HMY_KMI_THREADS) if (sSum[i] != 0.f) atomicAdd(&sums[i], (double)sSum[i]);
    for (int k = tid; k < K; k += HMY_KMI_THREADS) if (sCnt[k]) atomicAdd(&counts[k], sCnt[k]);
    if (lane == 0 && my_inertia != 0.0) atomicAdd(inertia, my_inertia);
}

// new centres = means (an empty cluster keeps its centre); info[0] = squared shift, info[1] = mean feature variance.
// n_cells: the number of cells the sums run over (all ranks' cells when the sums are global).
template <class CountT>
__device__ void lloyd_update(const HmyDev& st, float* C, const double* sums, const CountT* counts, double n_cells, double* info) {
    __shared__ double s_shift[32], s_mean2[32];
    const int K = st.K, dp = st.dp, d = st.d, tid = threadIdx.x;
    double shift = 0.0, mean2 = 0.0;
    for (int j = tid; j < d; j += blockDim.x) {                           // ||mean of all cells||^2, one feature per thread
        double s = 0.0;
        for (int k = 0; k < K; ++k) s += sums[(size_t)k * dp + j];
        s /= n_cells;
        mean2 += s * s;
    }
    for (int i = tid; i < K * dp; i += blockDim.x) {
        const int k = i / dp, j = i - k * dp;
        if (j < d && counts[k] > (CountT)0) {
            const float nc = (float)(sums[i] / (double)counts[k]);
            const double df = (double)nc - (double)C[i];
            shift += df * df;
            C[i] = nc;
        }
    }
    shift = warp_sum_d(shift); mean2 = warp_sum_d(mean2);
    if ((tid & 31) == 0) { s_shift[tid >> 5] = shift; s_mean2[tid >> 5] = mean2; }
    __syncthreads();
    if (tid == 0) {
        double a = 0.0, b = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a += s_shift[w]; b += s_mean2[w]; }
        info[0] = a;
        info[1] = (1.0 - b) / (double)d;                                  // rows of Z_cos have unit length: E|z|^2 = 1
    }
}

__global__ void k_lloyd_update(HmyDev st, float* C, const double* sums, const unsigned int* counts, double* info) {
    lloyd_update(st, C, sums, counts, (double)st.N, info);
}

// ---- cells sharded over ranks ----------------------------------------------------------------------------------------

// One seeding step on this rank's cells: D2 to centre c - 1 (row c - 1 of the gathered centres C), running minimum, race
// for centre c.  best[c] must be ~0ull on entry; afterwards it is {key bits, global id} of the local winner.
__global__ void __launch_bounds__(HMY_KMI_THREADS) k_kmpp_pass_sharded(HmyDev st, const float* C, int c, unsigned long long seed,
                                                                       float* mind2, unsigned long long* best) {
    extern __shared__ __align__(16) unsigned char kmi_smem[];
    float* sy = reinterpret_cast<float*>(kmi_smem);                       // [dp] the newest centre
    __shared__ unsigned long long s_best[HMY_KMI_THREADS / 32];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, dp = st.dp;
    for (int j = tid; j < dp; j += HMY_KMI_THREADS) sy[j] = C[(size_t)(c - 1) * dp + j];
    __syncthreads();
    unsigned long long mine = ~0ull;
    const long long nw = (long long)gridDim.x * (HMY_KMI_THREADS / 32);
    for (long long pos = (long long)blockIdx.x * (HMY_KMI_THREADS / 32) + warp; pos < st.N; pos += nw) {
        const float* z = st.Zcos + (size_t)pos * dp;
        float s = 0.f;
        for (int j = lane; j < dp; j += 32) { const float u = z[j] - sy[j]; s = fmaf(u, u, s); }
        s = warp_sum(s);
        if (lane == 0) {
            const float m = (c == 1) ? s : fminf(mind2[pos], s);
            mind2[pos] = m;
            if (m > 0.f) {
                const unsigned long long id = (unsigned long long)(st.cell_offset + st.order[pos]);   // < 2^32 (host check)
                const float key = (float)(-log(hmy_kmi_uniform(seed, c, id)) / (double)m);
                const unsigned long long packed = ((unsigned long long)__float_as_uint(key) << 32) | id;
                mine = packed < mine ? packed : mine;
            }
        }
    }
    if (lane == 0) s_best[warp] = mine;
    __syncthreads();
    if (tid == 0) {
        unsigned long long b = s_best[0];
        for (int w = 1; w < HMY_KMI_THREADS / 32; ++w) b = s_best[w] < b ? s_best[w] : b;
        if (b != ~0ull) atomicMin(&best[c], b);
    }
}

// This rank's candidate for centre c as slot `rank` of slots [world][2 + dp] = {key, global id, row}; every other slot
// is zeroed, so that the sum over ranks gathers all candidates exactly.  Centre 0 is cell first_id (key 0) on the rank
// that holds it; a rank without a candidate publishes key = +inf.
__global__ void k_kmpp_publish(HmyDev st, const unsigned long long* best, int c, long long first_id, int rank, int world,
                               double* slots) {
    const int dp = st.dp, S = 2 + dp;
    long long id = -1;
    double key = 0.0;
    if (c == 0) {
        if (first_id >= st.cell_offset && first_id < st.cell_offset + st.N) id = first_id;
    } else if (best[c] != ~0ull) {
        id = (long long)(best[c] & 0xFFFFFFFFull);
        key = (double)__uint_as_float((unsigned int)(best[c] >> 32));
    }
    const float* row = (id >= 0) ? st.Zcos + (size_t)st.pos_of[id - st.cell_offset] * dp : nullptr;
    for (int i = threadIdx.x; i < world * S; i += blockDim.x) {
        const int w = i / S, j = i - w * S;
        double v = 0.0;
        if (w == rank) v = (j == 0) ? (id >= 0 ? key : INFINITY) : (id < 0) ? 0.0 : (j == 1) ? (double)id : (double)row[j - 2];
        slots[i] = v;
    }
}

// Row c of the centres = the gathered candidate with the least (key, global id); *fail = 1 when no rank had one (no cell
// at a positive distance from the centres so far).
__global__ void k_kmpp_pick(const double* slots, int world, int dp, int c, float* C, int* fail) {
    __shared__ int s_w;
    const int S = 2 + dp;
    if (threadIdx.x == 0) {
        int bw = -1;
        for (int w = 0; w < world; ++w) {
            const double k = slots[(size_t)w * S], id = slots[(size_t)w * S + 1];
            if (!(k < INFINITY)) continue;
            if (bw < 0 || k < slots[(size_t)bw * S] || (k == slots[(size_t)bw * S] && id < slots[(size_t)bw * S + 1])) bw = w;
        }
        s_w = bw;
        if (bw < 0) *fail = 1;
    }
    __syncthreads();
    if (s_w < 0) return;
    for (int j = threadIdx.x; j < dp; j += blockDim.x) C[(size_t)c * dp + j] = (float)slots[(size_t)s_w * S + 2 + j];
}

// counts [K] -> the fp64 slice of the Lloyd table [sums K dp | counts K | inertia] that is summed over ranks
__global__ void k_lloyd_pack_counts(const unsigned int* counts, int K, double* tab_counts) {
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < K; k += gridDim.x * blockDim.x) tab_counts[k] = (double)counts[k];
}

// k_lloyd_update on the table summed over ranks.  info: [0] squared shift, [1] mean feature variance, [2] 1 if this rank
// would run another iteration (shift^2 > tol * variance), else 0, [3] global inertia.
__global__ void k_lloyd_update_global(HmyDev st, float* C, const double* tab, double tol, double* info) {
    const size_t nS = (size_t)st.K * st.dp;
    lloyd_update(st, C, tab, tab + nS, (double)st.Nglobal, info);
    if (threadIdx.x == 0) {
        info[2] = (info[0] <= tol * info[1]) ? 0.0 : 1.0;
        info[3] = tab[nS + st.K];
    }
}

// rank 0's centres (fp32 -> fp64), zeros on the other ranks: the sum over ranks hands everyone rank 0's centres exactly
__global__ void k_kmi_share(const float* C, size_t n, int keep, double* out) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = keep ? (double)C[i] : 0.0;
}

#endif  // HMY_NONTEMPLATE_KERNELS
