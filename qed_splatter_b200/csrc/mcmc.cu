// Splatfacto's MCMC densification strategy (nerfstudio 1.1.5 `strategy="mcmc"` -> gsplat 1.4.0 MCMCStrategy: relocate,
// sample_add, inject_noise_to_position, and splatfacto's two MCMC regularisers) on the flat arenas of trainer.GaussianArena
// (means 3N | quats 4N | log-scales 3N | logit-opacities N | SH 48N, each group 16-byte aligned; group starts passed as a
// host int64[5], as qed_arena_gather takes them).
//
// Sampling differs from gsplat on purpose: torch.multinomial's RNG stream cannot be reproduced, so draws come from a
// counter-based Philox4x32-10 (key = seed, counter = (draw index, step, stream id, 0)) through an inverse CDF over the
// exact int64 inclusive scan of the quantised weights floor(sigmoid(logit) * 2^24) (sigmoid in double).  Same inputs ->
// same draws on every rank, for any launch configuration; tests/mcmc_oracle.py restates it in numpy.
#include <cfloat>
#include <curand_philox4x32_x.h>

#include "common.cuh"
#include "scan.cuh"

namespace qed {

constexpr int kMcmcThreads = 256;
constexpr int kMcmcNMax = 51;          // gsplat's n_max: relocation ratios are clamped to [1, 51]
constexpr int kMcmcRegBlocks = 592;    // 148 SMs x 4: fixed upper bound of the regulariser grid (its partial sums)

struct McmcStarts {
    int64_t g[5];  // means, quats, log-scales, logit-opacities, SH
};

__device__ __forceinline__ float mcmc_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ uint4 mcmc_philox(uint64_t seed, uint32_t index, uint32_t step, uint32_t stream_id) {
    return curand_Philox4x32_10(make_uint4(index, step, stream_id, 0u), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}

// (0, 1] from 32 random bits, as curand's own uniform does it
__device__ __forceinline__ float mcmc_uniform(uint32_t x) { return (float)x * 2.3283064365386963e-10f + 1.1641532182693481e-10f; }

// scan input: 1 for a dead Gaussian (sigmoid(logit) <= min_opacity, decided in float32 as gsplat does)
struct McmcDeadFlag {
    const float* logit;
    float min_opacity;
    __device__ __forceinline__ int32_t operator()(int64_t i) const { return mcmc_sigmoid(logit[i]) <= min_opacity ? 1 : 0; }
};

// scan sink: the dead rows in ascending order (gsplat's mask.nonzero())
struct McmcCompact {
    int32_t* out;
    __device__ __forceinline__ void operator()(int64_t i, int32_t v, int64_t inc) const {
        if (v) out[inc - 1] = (int32_t)i;
    }
};

// scan input: quantised sampling weight floor(sigmoid(logit) * 2^24) <= 2^24, sigmoid in double; dead rows 0 when asked
struct McmcWeight {
    const float* logit;
    float min_opacity;
    int zero_dead;
    __device__ __forceinline__ int32_t operator()(int64_t i) const {
        const float x = logit[i];
        if (zero_dead && mcmc_sigmoid(x) <= min_opacity) return 0;
        return (int32_t)floor(16777216.0 / (1.0 + exp(-(double)x)));
    }
};

// draw j: u = (64 random bits * total) >> 64 in [0, total), row = first i with cum[i] > u.  cum[N-1] = total > u, so the
// search ends inside [0, N) and never on a row of zero weight.
__global__ void __launch_bounds__(kMcmcThreads) mcmc_draw_kernel(int64_t N, int64_t n_draws, const int64_t* __restrict__ cum,
                                                                const int64_t* __restrict__ total_dev, uint64_t seed, uint32_t step,
                                                                uint32_t stream_id, int32_t* __restrict__ draws, int32_t* __restrict__ counts) {
    pdl_enter();
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_draws) return;
    const uint64_t total = (uint64_t)*total_dev;
    if (total == 0) return;  // nothing to draw from (torch.multinomial would raise): draws untouched, counts stay zero
    const uint4 r = mcmc_philox(seed, (uint32_t)j, step, stream_id);
    const uint64_t u = __umul64hi(((uint64_t)r.x << 32) | r.y, total);
    int64_t lo = 0, hi = N - 1;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if ((uint64_t)cum[mid] > u) hi = mid;
        else lo = mid + 1;
    }
    draws[j] = (int32_t)lo;
    atomicAdd(counts + lo, 1);  // integer: the same counts whatever the order
}

// gsplat compute_relocation for a row drawn c = counts[i] times (ratio n = min(c + 1, 51)), in place:
//   o' = 1 - (1 - o)^(1/n),  scale' = o / D(o', n) * scale,  D(x, n) = sum_{j=1..n} C(n, j) (-1)^(j-1) x^j / sqrt(j)
// D is gsplat's double loop sum_{i=1..n} sum_{k<i} C(i-1, k) (-1)^k x^(k+1) / sqrt(k+1) folded by the hockey-stick
// identity sum_{i=k+1..n} C(i-1, k) = C(n, k+1), and evaluated in float64 (gsplat's float32 loop loses ~5e-4 to
// cancellation at n = 51).  o' is clamped to [min_opacity, 1 - FLT_EPSILON] after the scale uses it, as in gsplat.
// Every thread reads and writes only its own row: rows drawn several times are updated once, from their old values.
__global__ void __launch_bounds__(kMcmcThreads) mcmc_relocation_kernel(int64_t N, const int32_t* __restrict__ counts, float min_opacity,
                                                                      int zero_moments, float* __restrict__ p, float* __restrict__ m,
                                                                      float* __restrict__ v, McmcStarts st) {
    pdl_enter();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int c = counts[i];
    if (c <= 0) return;
    const int n = min(c + 1, kMcmcNMax);
    float* op = p + st.g[3] + i;
    const double o = (double)mcmc_sigmoid(*op);
    const double x = 1.0 - pow(1.0 - o, 1.0 / (double)n);
    double binom = 1.0, xp = 1.0, D = 0.0;
    for (int j = 1; j <= n; ++j) {
        binom = binom * (double)(n - j + 1) / (double)j;  // C(n, j), exact in float64 for n <= 51
        xp *= x;
        const double t = binom * xp / sqrt((double)j);
        D += (j & 1) ? t : -t;
    }
    const double coeff = o / D;
    const float on = fminf(fmaxf((float)x, min_opacity), 1.0f - FLT_EPSILON);
    *op = logf(on / (1.0f - on));
    float* ls = p + st.g[2] + i * 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) ls[k] = logf((float)(coeff * (double)expf(ls[k])));
    if (zero_moments) {
        const int dims[5] = {3, 4, 3, 1, 48};
#pragma unroll
        for (int g = 0; g < 5; ++g)
            for (int k = 0; k < dims[g]; ++k) {
                m[st.g[g] + i * dims[g] + k] = 0.0f;
                v[st.g[g] + i * dims[g] + k] = 0.0f;
            }
    }
}

// relocate's second half: parameter row src[j] -> row dst[j] (moments of dst untouched).  16 lanes per copy: lanes 0..11 the
// SH row (12 x float4), lanes 12..15 means / quats / log-scales / logit-opacity.  Sources and destinations are disjoint
// (drawn rows are alive, destinations dead), so no row is read and written in the same launch.
__global__ void __launch_bounds__(kMcmcThreads) mcmc_copy_rows_kernel(int64_t n, const int32_t* __restrict__ src, const int32_t* __restrict__ dst,
                                                                     float* __restrict__ p, McmcStarts st) {
    pdl_enter();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t j = t >> 4;
    const int l = (int)(t & 15);
    if (j >= n) return;
    const int64_t s = src[j], d = dst[j];
    if (l < 12) {
        *reinterpret_cast<float4*>(p + st.g[4] + d * 48 + l * 4) = *reinterpret_cast<const float4*>(p + st.g[4] + s * 48 + l * 4);
        return;
    }
    const int grp = l - 12;
    const int dim = grp == 1 ? 4 : (grp == 3 ? 1 : 3);
    const int64_t g0 = grp == 0 ? st.g[0] : (grp == 1 ? st.g[1] : (grp == 2 ? st.g[2] : st.g[3]));  // no dynamic index: no stack frame
    for (int k = 0; k < dim; ++k) p[g0 + d * dim + k] = p[g0 + s * dim + k];
}

// gsplat inject_noise_to_position: means += R diag(s)^2 R^T (n * sigmoid(100 ((1 - o) - 0.995)) * scaler), n ~ N(0, I_3)
// from Box-Muller on Philox counter (i, step, 0, 0) (three of its four normals); R from the normalised quaternion (w, x, y, z).
__global__ void __launch_bounds__(kMcmcThreads) mcmc_noise_kernel(int64_t N, float* __restrict__ p, McmcStarts st, float scaler, uint64_t seed,
                                                                 uint32_t step) {
    pdl_enter();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const float4 q = *reinterpret_cast<const float4*>(p + st.g[1] + i * 4);
    const float qn = 1.0f / fmaxf(sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w), 1e-12f);
    const float w = q.x * qn, x = q.y * qn, y = q.z * qn, z = q.w * qn;
    const float R[3][3] = {{1.f - 2.f * (y * y + z * z), 2.f * (x * y - w * z), 2.f * (x * z + w * y)},
                           {2.f * (x * y + w * z), 1.f - 2.f * (x * x + z * z), 2.f * (y * z - w * x)},
                           {2.f * (x * z - w * y), 2.f * (y * z + w * x), 1.f - 2.f * (x * x + y * y)}};
    const float* ls = p + st.g[2] + i * 3;
    float s2[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float s = expf(ls[k]);
        s2[k] = s * s;
    }
    const float o = mcmc_sigmoid(p[st.g[3] + i]);
    const float f = scaler / (1.0f + expf(-100.0f * ((1.0f - o) - 0.995f)));
    const uint4 r = mcmc_philox(seed, (uint32_t)i, step, 0u);
    float sn, cs, sn2, cs2;
    sincospif(2.0f * mcmc_uniform(r.y), &sn, &cs);
    sincospif(2.0f * mcmc_uniform(r.w), &sn2, &cs2);
    const float r1 = sqrtf(-2.0f * logf(mcmc_uniform(r.x))), r2 = sqrtf(-2.0f * logf(mcmc_uniform(r.z)));
    const float nv[3] = {r1 * cs * f, r1 * sn * f, r2 * cs2 * f};
    float u[3];  // diag(s^2) R^T n
#pragma unroll
    for (int k = 0; k < 3; ++k) u[k] = s2[k] * (R[0][k] * nv[0] + R[1][k] * nv[1] + R[2][k] * nv[2]);
    float* mu = p + st.g[0] + i * 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) mu[k] += R[k][0] * u[0] + R[k][1] * u[1] + R[k][2] * u[2];
}

// splatfacto's MCMC regularisers: loss[0] = opacity_reg * mean_N sigmoid(logit), loss[1] = scale_reg * mean_3N exp(log-scale);
// their gradients are added to the gradient arena.  Per-block float64 partial sums, summed in block order by the last block
// to finish (a ticket in the workspace, left at zero): the same inputs give the same bits on every rank.
__global__ void __launch_bounds__(kMcmcThreads) mcmc_reg_kernel(int64_t N, const float* __restrict__ p, float* __restrict__ grad, McmcStarts st,
                                                               float opacity_reg, float scale_reg, double* __restrict__ partials,
                                                               unsigned int* __restrict__ ticket, float* __restrict__ loss) {
    __shared__ double s_a[kMcmcThreads / 32], s_b[kMcmcThreads / 32];
    __shared__ bool s_last;
    pdl_enter();
    const float go = (float)((double)opacity_reg / (double)N), gs = (float)((double)scale_reg / (3.0 * (double)N));
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    double a = 0.0, b = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
        const float o = mcmc_sigmoid(p[st.g[3] + i]);
        grad[st.g[3] + i] += go * (o * (1.0f - o));
        a += (double)o;
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < 3 * N; i += stride) {
        const float e = expf(p[st.g[2] + i]);
        grad[st.g[2] + i] += gs * e;
        b += (double)e;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if ((threadIdx.x & 31) == 0) {
        s_a[threadIdx.x >> 5] = a;
        s_b[threadIdx.x >> 5] = b;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kMcmcThreads / 32; ++w) {
            a += s_a[w];
            b += s_b[w];
        }
        partials[2 * blockIdx.x] = a;
        partials[2 * blockIdx.x + 1] = b;
        __threadfence();
        s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last || threadIdx.x != 0) return;
    __threadfence();
    double sa = 0.0, sb = 0.0;
    for (unsigned int k = 0; k < gridDim.x; ++k) {
        sa += reinterpret_cast<volatile double*>(partials)[2 * k];
        sb += reinterpret_cast<volatile double*>(partials)[2 * k + 1];
    }
    loss[0] = (float)((double)opacity_reg * sa / (double)N);
    loss[1] = (float)((double)scale_reg * sb / (3.0 * (double)N));
    *ticket = 0u;
}

inline McmcStarts mcmc_starts(const int64_t* g) {
    McmcStarts s;
    for (int k = 0; k < 5; ++k) s.g[k] = g[k];
    return s;
}

inline size_t mcmc_align16(size_t b) { return (b + 15) / 16 * 16; }

}  // namespace qed

using namespace qed;

extern "C" size_t qed_mcmc_workspace_bytes(int64_t N) {
    if (N < 0) return 0;
    return mcmc_align16((size_t)N * sizeof(int64_t)) + scan_workspace_bytes(N);
}

extern "C" int qed_mcmc_census(int64_t N, const float* logit_opacities, float min_opacity, int32_t* dead_idx, int64_t* n_dead_dev, void* workspace,
                               size_t workspace_bytes, qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (N < 0 || N > 0x7fffffffLL) return N < 0 ? QED_ERR_BAD_ARG : QED_ERR_UNSUPPORTED;
    if (!n_dead_dev) return QED_ERR_BAD_ARG;
    if (N == 0) {
        QED_CUDA_TRY(cudaMemsetAsync(n_dead_dev, 0, sizeof(int64_t), stream));
        return QED_OK;
    }
    if (!logit_opacities || !dead_idx || !workspace) return QED_ERR_BAD_ARG;
    if (workspace_bytes < qed_mcmc_workspace_bytes(N)) return QED_ERR_WORKSPACE;
    return scan_inclusive_to(N, nullptr, McmcDeadFlag{logit_opacities, min_opacity}, McmcCompact{dead_idx}, n_dead_dev,
                             reinterpret_cast<char*>(workspace) + mcmc_align16((size_t)N * sizeof(int64_t)), stream);
}

extern "C" int qed_mcmc_sample(int64_t N, const float* logit_opacities, float min_opacity, int zero_dead, int64_t n_draws, uint64_t seed, uint32_t step,
                               uint32_t stream_id, int32_t* draws, int32_t* counts, int64_t* total_dev, void* workspace, size_t workspace_bytes,
                               qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (N < 0 || n_draws < 0) return QED_ERR_BAD_ARG;
    if (N > 0x7fffffffLL || n_draws > 0x7fffffffLL) return QED_ERR_UNSUPPORTED;
    if (!total_dev) return QED_ERR_BAD_ARG;
    if (N == 0) {
        QED_CUDA_TRY(cudaMemsetAsync(total_dev, 0, sizeof(int64_t), stream));
        return QED_OK;
    }
    if (!logit_opacities || !counts || !workspace || (n_draws > 0 && !draws)) return QED_ERR_BAD_ARG;
    if (workspace_bytes < qed_mcmc_workspace_bytes(N)) return QED_ERR_WORKSPACE;
    int64_t* cum = reinterpret_cast<int64_t*>(workspace);
    void* scan_ws = reinterpret_cast<char*>(workspace) + mcmc_align16((size_t)N * sizeof(int64_t));
    QED_CUDA_TRY(cudaMemsetAsync(counts, 0, (size_t)N * sizeof(int32_t), stream));
    int rc = scan_inclusive(N, nullptr, McmcWeight{logit_opacities, min_opacity, zero_dead ? 1 : 0}, cum, total_dev, scan_ws, stream);
    if (rc != QED_OK) return rc;
    if (n_draws == 0) return QED_OK;
    QED_CUDA_TRY(launch_pdl(mcmc_draw_kernel, dim3((unsigned)((n_draws + kMcmcThreads - 1) / kMcmcThreads)), dim3(kMcmcThreads), 0, stream, N, n_draws,
                            (const int64_t*)cum, (const int64_t*)total_dev, seed, step, stream_id, draws, counts));
    return QED_OK;
}

extern "C" int qed_mcmc_relocate(int64_t N, const int32_t* counts, float min_opacity, int zero_moments, int64_t n_copies, const int32_t* src,
                                 const int32_t* dst, float* param, float* exp_avg, float* exp_avg_sq, const int64_t* group_starts,
                                 qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (N < 0 || n_copies < 0) return QED_ERR_BAD_ARG;
    if (N > 0x7fffffffLL || n_copies > 0x7fffffffLL) return QED_ERR_UNSUPPORTED;
    if (N == 0) return QED_OK;
    if (!counts || !param || !group_starts || (zero_moments && (!exp_avg || !exp_avg_sq)) || (n_copies > 0 && (!src || !dst)))
        return QED_ERR_BAD_ARG;
    const McmcStarts st = mcmc_starts(group_starts);
    if ((st.g[1] & 3) || (st.g[4] & 3) || (reinterpret_cast<uintptr_t>(param) & 15)) return QED_ERR_BAD_ARG;  // float4 rows
    QED_CUDA_TRY(launch_pdl(mcmc_relocation_kernel, dim3((unsigned)((N + kMcmcThreads - 1) / kMcmcThreads)), dim3(kMcmcThreads), 0, stream, N, counts,
                            min_opacity, zero_moments ? 1 : 0, param, exp_avg, exp_avg_sq, st));
    if (n_copies > 0)
        QED_CUDA_TRY(launch_pdl(mcmc_copy_rows_kernel, dim3((unsigned)((n_copies * 16 + kMcmcThreads - 1) / kMcmcThreads)), dim3(kMcmcThreads), 0, stream,
                                n_copies, src, dst, param, st));
    return QED_OK;
}

extern "C" int qed_mcmc_noise(int64_t N, float* param, const int64_t* group_starts, float scaler, uint64_t seed, uint32_t step, qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (N < 0) return QED_ERR_BAD_ARG;
    if (N > 0x7fffffffLL) return QED_ERR_UNSUPPORTED;
    if (N == 0) return QED_OK;
    if (!param || !group_starts) return QED_ERR_BAD_ARG;
    const McmcStarts st = mcmc_starts(group_starts);
    if ((st.g[1] & 3) || (reinterpret_cast<uintptr_t>(param) & 15)) return QED_ERR_BAD_ARG;
    QED_CUDA_TRY(launch_pdl(mcmc_noise_kernel, dim3((unsigned)((N + kMcmcThreads - 1) / kMcmcThreads)), dim3(kMcmcThreads), 0, stream, N, param, st,
                            scaler, seed, step));
    return QED_OK;
}

extern "C" size_t qed_mcmc_reg_workspace_bytes(void) { return (size_t)kMcmcRegBlocks * 2 * sizeof(double) + 16; }

extern "C" int qed_mcmc_reg(int64_t N, const float* param, const int64_t* group_starts, float opacity_reg, float scale_reg, float* grad, float* loss,
                            void* workspace, size_t workspace_bytes, qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (N <= 0 || !param || !group_starts || !grad || !loss || !workspace) return QED_ERR_BAD_ARG;
    if (workspace_bytes < qed_mcmc_reg_workspace_bytes()) return QED_ERR_WORKSPACE;
    const McmcStarts st = mcmc_starts(group_starts);
    const int64_t need = (N + kMcmcThreads - 1) / kMcmcThreads;
    const unsigned blocks = (unsigned)(need < kMcmcRegBlocks ? need : kMcmcRegBlocks);
    double* partials = reinterpret_cast<double*>(workspace);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(partials + 2 * kMcmcRegBlocks);
    QED_CUDA_TRY(launch_pdl(mcmc_reg_kernel, dim3(blocks), dim3(kMcmcThreads), 0, stream, N, param, grad, st, opacity_reg, scale_reg, partials, ticket,
                            loss));
    return QED_OK;
}
