// Splatfacto's resolution schedule on the data side: the ground truth of a step rendered at 1/d resolution is reduced by
// nerfstudio's `resize_image` (splatfacto `_downscale_if_required`: conv2d with a d x d kernel of weights 1/d^2 and
// stride d) applied to the image, the depth and `batch["mask"]`.  One pass reads the full-resolution cache in its stored
// type (uint8 image, raw uint16 depth, bool mask), converts each value exactly as the loss kernels do (GtImage /
// GtDepth / PixelMask) and writes the float32 ground truth the loss reads at render size.
#include "common.cuh"

namespace qed {

// One thread per output pixel.  Each output is the sum over its d x d block, in row-major order starting from 0, of
// (1/d^2) * x with individually rounded IEEE ops (no FMA), so the result is a fixed function of the inputs.
__global__ void downscale_gt_kernel(int64_t n_out, int w, int h, int width, int height, int d, float inv, GtImage rgb, GtDepth depth,
                                    PixelMask mask, float* __restrict__ out_rgb, float* __restrict__ out_depth, float* __restrict__ out_mask) {
    pdl_enter();
    const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n_out) return;
    const int64_t hw = (int64_t)h * w;
    const int64_t c = o / hw;
    const int rem = (int)(o - c * hw);
    const int y = rem / w, x = rem - (rem / w) * w;
    const int64_t base = (c * height + (int64_t)y * d) * width + (int64_t)x * d;
    float r = 0.0f, g = 0.0f, b = 0.0f, z = 0.0f, m = 0.0f;
    for (int dy = 0; dy < d; ++dy) {
        const int64_t row = base + (int64_t)dy * width;
        for (int dx = 0; dx < d; ++dx) {
            const int64_t pix = row + dx;
            r = add(r, mul(inv, rgb.at(pix * 3 + 0)));
            g = add(g, mul(inv, rgb.at(pix * 3 + 1)));
            b = add(b, mul(inv, rgb.at(pix * 3 + 2)));
            z = add(z, mul(inv, depth.at(pix)));
            if (out_mask) m = add(m, mul(inv, mask.at(pix)));
        }
    }
    out_rgb[o * 3 + 0] = r;
    out_rgb[o * 3 + 1] = g;
    out_rgb[o * 3 + 2] = b;
    out_depth[o] = z;
    if (out_mask) out_mask[o] = m;
}

}  // namespace qed

using namespace qed;

extern "C" int qed_downscale_ground_truth(int C, int width, int height, int factor, const void* gt_rgb, int rgb_is_u8, const void* gt_depth,
                                          int depth_is_u16, double depth_unit_scale, const void* mask, int mask_is_u8, float* out_rgb,
                                          float* out_depth, float* out_mask, qed_stream_t stream) {
    if (C < 1 || width < 1 || height < 1 || factor < 1) return QED_ERR_BAD_ARG;
    const int w = width / factor, h = height / factor;
    if (w == 0 || h == 0) return QED_ERR_BAD_ARG;
    if (!gt_rgb || !gt_depth || !out_rgb || !out_depth || (mask && !out_mask)) return QED_ERR_BAD_ARG;
    const int64_t n_out = (int64_t)C * h * w;
    const float inv = 1.0f / (float)((int64_t)factor * factor);
    QED_CUDA_TRY(launch_pdl(downscale_gt_kernel, dim3((unsigned)((n_out + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, n_out, w, h, width,
                            height, factor, inv, GtImage{gt_rgb, rgb_is_u8}, GtDepth{gt_depth, depth_is_u16, depth_unit_scale},
                            PixelMask{mask, mask_is_u8}, out_rgb, out_depth, mask ? out_mask : nullptr));
    return QED_OK;
}
