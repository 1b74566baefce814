// Held-out evaluation metrics: PSNR, SSIM and the depth metrics of qed-splatter's DepthMetrics (metrics.py:115-156) per view.
//
// Forward only, three launches, no float atomics:
//   eval_fill_kernel    per-view maximum of the rendered depth (the fill value of model.py:304-306, as loss_stats_kernel
//                       finds it: max over every pixel, starting at 0; integer atomicMax on the float bits, so any order
//                       gives the same value);
//   ssim_fwd_kernel<true> (ssim.cu)  per-block partials of the SSIM map, the squared RGB error and the depth sums;
//   eval_finalize_kernel one block per view sums its partials in a fixed order and writes the view's row.
// The same inputs give the same bits, and a view's row does not depend on the other views of the batch.
#include "common.cuh"

namespace qed {

constexpr int kFillThreads = 256;
constexpr int kFillUnroll = 4;
constexpr int kFinalizeThreads = 256;

__global__ void __launch_bounds__(kFillThreads) eval_fill_kernel(int64_t HW, const float4* __restrict__ render, int* __restrict__ fill) {
    pdl_enter();
    const int cam = blockIdx.y;
    float maxd = 0.0f;
    const int64_t base = (int64_t)blockIdx.x * (kFillThreads * kFillUnroll) + threadIdx.x;
#pragma unroll
    for (int u = 0; u < kFillUnroll; ++u) {
        const int64_t i = base + (int64_t)u * kFillThreads;
        if (i < HW) maxd = fmaxf(maxd, render[cam * HW + i].w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) maxd = fmaxf(maxd, __shfl_xor_sync(0xffffffffu, maxd, o));
    if ((threadIdx.x & 31) == 0) atomicMax(fill + cam, __float_as_int(maxd));  // >= +0.0f: int order = float order
}

// one block per view: thread t sums tiles t, t + 256, ... of the three channels in order, then xor shuffles and the warps in order
__global__ void __launch_bounds__(kFinalizeThreads) eval_finalize_kernel(int64_t tiles, int W, int H, const double* __restrict__ partials,
                                                                       double* __restrict__ metrics) {
    __shared__ double red[kFinalizeThreads / 32][kEvalPartials];
    pdl_enter();
    const int cam = blockIdx.x;
    double s[kEvalPartials] = {};
    for (int ch = 0; ch < 3; ++ch) {
        const double* p = partials + ((int64_t)cam * 3 + ch) * tiles * kEvalPartials;
        for (int64_t t = threadIdx.x; t < tiles; t += kFinalizeThreads)
#pragma unroll
            for (int k = 0; k < kEvalPartials; ++k) s[k] += p[t * kEvalPartials + k];
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < kEvalPartials; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
        if (lane == 0) red[warp][k] = s[k];
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    double t[kEvalPartials];
    for (int k = 0; k < kEvalPartials; ++k) {
        t[k] = red[0][k];
        for (int w = 1; w < kFinalizeThreads / 32; ++w) t[k] += red[w][k];
    }
    const double mse = t[1] / ((double)W * (double)H * 3.0);
    const double n = t[2];  // n == 0: every depth mean below is 0 / 0 = NaN, as torch's mean of an empty tensor
    double* m = metrics + (int64_t)cam * QED_EVAL_METRICS;
    m[0] = 10.0 * log10(1.0 / mse);  // a perfect image: +inf
    m[1] = t[0] / ((double)(W - 10) * (double)(H - 10) * 3.0);
    m[2] = mse;
    m[3] = t[3] / n;
    m[4] = t[4] / n;
    m[5] = sqrt(t[5] / n);
    m[6] = sqrt(t[6] / n);
    m[7] = t[7] / n;
    m[8] = t[8] / n;
    m[9] = t[9] / n;
    m[10] = n;
}

static size_t fill_bytes(int C) { return ((size_t)C * sizeof(int) + 255) / 256 * 256; }

}  // namespace qed

using namespace qed;

int64_t qed_ssim_eval_tiles(int W, int H);  // ssim.cu
int qed_ssim_eval_launch(int C, int W, int H, const float* render, const float* alphas, qed::GtImage gt, qed::GtDepth gt_depth, const float* bg,
                         const int* fill, float depth_tol, double* partials, cudaStream_t stream);  // ssim.cu

extern "C" size_t qed_eval_metrics_workspace_bytes(int C, int width, int height) {
    if (C <= 0 || width <= 10 || height <= 10) return 0;
    return fill_bytes(C) + (size_t)C * 3 * (size_t)qed_ssim_eval_tiles(width, height) * kEvalPartials * sizeof(double);
}

extern "C" int qed_eval_metrics(int C, int width, int height, const float* render, const float* alphas, const void* gt_rgb, int gt_rgb_is_u8,
                                const void* gt_depth, int gt_depth_is_u16, double depth_unit_scale, const float* bg, float depth_tolerance,
                                double* metrics_dev, void* workspace, size_t workspace_bytes, qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (C <= 0 || width <= 0 || height <= 0) return QED_ERR_BAD_ARG;
    if (!render || !alphas || !gt_rgb || !gt_depth || !bg || !metrics_dev || !workspace) return QED_ERR_BAD_ARG;
    if (width <= 10 || height <= 10 || C > 21845) return QED_ERR_UNSUPPORTED;  // SSIM's valid windows; grid.z = 3 C
    if (workspace_bytes < qed_eval_metrics_workspace_bytes(C, width, height)) return QED_ERR_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(workspace) & 15) return QED_ERR_BAD_ARG;
    const int64_t HW = (int64_t)width * height;
    int* fill = reinterpret_cast<int*>(workspace);
    double* partials = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + fill_bytes(C));
    QED_CUDA_TRY(cudaMemsetAsync(fill, 0, (size_t)C * sizeof(int), stream));
    const int bx = (int)((HW + kFillThreads * kFillUnroll - 1) / (kFillThreads * kFillUnroll));
    QED_CUDA_TRY(launch_pdl(eval_fill_kernel, dim3(bx, C), dim3(kFillThreads), 0, stream, HW, reinterpret_cast<const float4*>(render), fill));
    const GtImage gi{gt_rgb, gt_rgb_is_u8 ? 1 : 0};
    const GtDepth gd{gt_depth, gt_depth_is_u16 ? 1 : 0, depth_unit_scale};
    int rc = qed_ssim_eval_launch(C, width, height, render, alphas, gi, gd, bg, fill, depth_tolerance, partials, stream);
    if (rc != QED_OK) return rc;
    QED_CUDA_TRY(launch_pdl(eval_finalize_kernel, dim3(C), dim3(kFinalizeThreads), 0, stream, qed_ssim_eval_tiles(width, height), width, height,
                            (const double*)partials, metrics_dev));
    return QED_OK;
}
