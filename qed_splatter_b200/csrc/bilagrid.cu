// Trainer-side kernels of splatfacto's bilateral grid (nerfstudio lib_bilagrid): the total-variation regulariser over all
// grids and the sum of per-view gradient rows into the dense grid gradient.  The slice itself is fused into the loss
// (train.cu, qed_loss_fwd_bwd_bilagrid).
#include "common.cuh"

namespace qed {

constexpr int kTvThreads = 256;

// One block per grid: each element's gradient is gathered from its (up to 6) neighbours, so nothing is accumulated across
// threads; the grid's sums of squared differences per axis are reduced in a fixed order in float64 and summed over the grids
// by bilagrid_tv_finish_kernel.  32-bit index arithmetic (a grid has < 2^31 elements; the entry point checks the whole table).
// tv = weight / G * sum_axes sum (x[i+1] - x[i])^2 / (12 L Y X (n_axis - 1) / n_axis).
__global__ void __launch_bounds__(kTvThreads) bilagrid_tv_kernel(int X, int Y, int L, const float* __restrict__ grids, float weight, int G,
                                                                float* __restrict__ v_grids, double* __restrict__ partials) {
    __shared__ double part[kTvThreads / 32];
    pdl_enter();
    const int sz = X * Y, n = sz * L * 12;
    const float* g = grids + (int64_t)blockIdx.x * n;
    float* v = v_grids + (int64_t)blockIdx.x * n;
    // per-axis coefficient of d/dx (x[i+1]-x[i])^2 / count: 2 / count, times weight / G
    const double cnt_x = 12.0 * L * Y * (X - 1), cnt_y = 12.0 * L * (Y - 1) * X, cnt_z = 12.0 * (L - 1) * Y * X;
    const float kx = (float)(2.0 * weight / G / cnt_x), ky = (float)(2.0 * weight / G / cnt_y), kz = (float)(2.0 * weight / G / cnt_z);
    double acc_x = 0.0, acc_y = 0.0, acc_z = 0.0;
    for (int p = 0; p < 12 * L; ++p) {  // [Y, X] planes in order; z = level of the plane
        const int z = p % L, base = p * sz;
        for (int e = threadIdx.x; e < sz; e += kTvThreads) {
            const int x = e % X, y = e / X, i = base + e;
            const float c = g[i];
            float gr = 0.0f;
            if (x > 0) gr += kx * (c - g[i - 1]);
            if (x < X - 1) {
                const float d = g[i + 1] - c;
                gr -= kx * d;
                acc_x += (double)d * d;
            }
            if (y > 0) gr += ky * (c - g[i - X]);
            if (y < Y - 1) {
                const float d = g[i + X] - c;
                gr -= ky * d;
                acc_y += (double)d * d;
            }
            if (z > 0) gr += kz * (c - g[i - sz]);
            if (z < L - 1) {
                const float d = g[i + sz] - c;
                gr -= kz * d;
                acc_z += (double)d * d;
            }
            v[i] = gr;
        }
    }
    double acc = acc_x / cnt_x + acc_y / cnt_y + acc_z / cnt_z;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = part[0];
        for (int w = 1; w < kTvThreads / 32; ++w) s += part[w];
        partials[blockIdx.x] = s;
    }
}

__global__ void __launch_bounds__(kTvThreads) bilagrid_tv_finish_kernel(int n, int G, float weight, const double* __restrict__ partials, float* __restrict__ loss) {
    __shared__ double part[kTvThreads / 32];
    pdl_enter();
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += kTvThreads) acc += partials[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = part[0];
        for (int w = 1; w < kTvThreads / 32; ++w) s += part[w];
        *loss = (float)((double)weight * s / G);
    }
}

// v_grids[ids[r]] += v_rows[r] for r = 0..n_rows-1 in row order (one thread per element of a row): views that share a grid
// are summed in view order, deterministically.  Rows with an id outside [0, G) are skipped.
__global__ void __launch_bounds__(256) bilagrid_accumulate_kernel(int n_rows, const int32_t* __restrict__ ids, int64_t row, const float* __restrict__ v_rows,
                                                                  int G, float* __restrict__ v_grids) {
    pdl_enter();
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= row) return;
    for (int r = 0; r < n_rows; ++r) {
        const int g = ids[r];
        if (g < 0 || g >= G) continue;
        v_grids[(int64_t)g * row + e] += v_rows[(int64_t)r * row + e];
    }
}

}  // namespace qed

using namespace qed;

static bool bilagrid_shape_ok(int X, int Y, int L) { return X >= 2 && Y >= 2 && L >= 2 && X <= 1024 && Y <= 1024 && L <= 16; }

extern "C" int qed_bilagrid_tv(int num_grids, int grid_X, int grid_Y, int grid_L, const float* grids, float weight, float* v_grids,
                               double* tv_per_grid, float* loss_out, qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (num_grids <= 0 || !grids || !v_grids || !tv_per_grid || !loss_out) return QED_ERR_BAD_ARG;
    if (!bilagrid_shape_ok(grid_X, grid_Y, grid_L) || num_grids > 0x7fffffff / 12 / (grid_X * grid_Y * grid_L)) return QED_ERR_UNSUPPORTED;
    QED_CUDA_TRY(launch_pdl(bilagrid_tv_kernel, dim3((unsigned)num_grids), dim3(kTvThreads), 0, stream, grid_X, grid_Y, grid_L, grids, weight,
                            num_grids, v_grids, tv_per_grid));
    QED_CUDA_TRY(launch_pdl(bilagrid_tv_finish_kernel, dim3(1), dim3(kTvThreads), 0, stream, num_grids, num_grids, weight,
                            (const double*)tv_per_grid, loss_out));
    return QED_OK;
}

extern "C" int qed_bilagrid_accumulate(int n_rows, const int32_t* grid_ids, const float* v_grid_rows, int num_grids, int grid_X, int grid_Y,
                                       int grid_L, float* v_grids, qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n_rows < 0 || num_grids <= 0) return QED_ERR_BAD_ARG;
    if (n_rows == 0) return QED_OK;
    if (!grid_ids || !v_grid_rows || !v_grids) return QED_ERR_BAD_ARG;
    if (!bilagrid_shape_ok(grid_X, grid_Y, grid_L)) return QED_ERR_UNSUPPORTED;
    const int64_t row = (int64_t)12 * grid_X * grid_Y * grid_L;
    QED_CUDA_TRY(launch_pdl(bilagrid_accumulate_kernel, dim3((unsigned)((row + 255) / 256)), dim3(256), 0, stream, n_rows, grid_ids, row, v_grid_rows,
                            num_grids, v_grids));
    return QED_OK;
}
