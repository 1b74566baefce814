// SSIM (11x11 Gaussian window, sigma 1.5, "valid" convolution) forward + backward, fused.
//
// This is the `1 - SSIM` term of splatfacto's RGB loss, reached from qed_splatter/model.py:83-85
// (nerfstudio: pytorch_msssim.SSIM(data_range=1.0, size_average=True, channel=3)); SURVEY.md §8f#1.
// Semantics == oracle/torch_impl.py::ssim.  X = ground truth, Y = prediction, per channel:
//   mu = w*X, w*Y ; e = w*X^2, w*Y^2, w*XY ; s1 = e1 - mu1^2, s2 = e2 - mu2^2, s12 = e12 - mu1 mu2
//   map = (2 mu1 mu2 + C1)(2 s12 + C2) / ((mu1^2 + mu2^2 + C1)(s1 + s2 + C2)),  C1 = 0.01^2, C2 = 0.03^2
// forward kernel : one CTA per 32x32 tile of the valid output, separable 11-tap filter in shared memory (register sliding
//                  windows, two adjacent outputs per FFMA2: the weight pair (w[k], w[k-1]) times a broadcast input), writes
//                  the three partial-derivative maps d map/d(mu2, e2, e12) and accumulates sum(map).
//                  Its EVAL instantiation (held-out metrics, metrics.cu) forms the prediction from the render itself and
//                  writes per-block partial sums instead (see SsimEval).
// backward kernel: dL/dY(p) = sum_q w(q-p) [Dmu(q) + 2 Y(p) De2(q) + X(p) De12(q)] * scale  (zero outside the
//                  valid region), again separable.  HBM-bound: ~15 floats per pixel-channel moved in total.
#include "common.cuh"

namespace qed {

constexpr int kWin = 11;
constexpr int kHalo = kWin - 1;
constexpr int kSsimTile = 32;               // outputs per CTA: 32 x 32
constexpr int kSsimIn = kSsimTile + kHalo;  // 42
constexpr int kBlkH = 8;                    // outputs per thread of the horizontal pass (register sliding window)
constexpr int kBlkV = 4;                    // outputs per thread of the vertical pass
constexpr int kHStride = kSsimTile + 2;     // row stride of the horizontally filtered planes: even, so pairs store as 64 bits
constexpr int kSsimThreads = 256;

// w[k]: the 11 taps (symmetric).  p[k] = (w[k], w[k-1]) with w[-1] = w[11] = 0: the weight pair of input tap t for the two
// adjacent outputs (o, o+1), k = t - o -- one FFMA2 with a scalar-broadcast input updates both.
struct GaussWin {
    float w[kWin];
    float pad_;
    float2 p[kWin + 1];
};

static GaussWin make_window() {
    GaussWin g;
    double s = 0.0, v[kWin];
    for (int i = 0; i < kWin; ++i) {
        const double c = i - kWin / 2;
        v[i] = exp(-(c * c) / (2.0 * 1.5 * 1.5));
        s += v[i];
    }
    for (int i = 0; i < kWin; ++i) g.w[i] = (float)(v[i] / s);
    for (int i = 0; i < kWin / 2; ++i) g.w[kWin - 1 - i] = g.w[i];  // exactly symmetric (the backward filter is the mirrored one)
    g.pad_ = 0.0f;
    for (int k = 0; k <= kWin; ++k) g.p[k] = make_float2(k < kWin ? g.w[k] : 0.0f, k > 0 ? g.w[k - 1] : 0.0f);
    return g;
}

// Separable 11-tap filter of NQ planes, NB outputs per thread from a register sliding window, two outputs per FFMA2.
// `load(t, v)` fills v[0..NQ) with the NQ inputs at tap t (t = 0 .. kWin + NB - 2); acc2[q][j] = outputs (2j, 2j+1) of plane q.
template <int NQ, int NB, typename Load>
__device__ __forceinline__ void filter_taps(const GaussWin& win, f32x2 (&acc2)[NQ][NB / 2], Load load) {
#pragma unroll
    for (int q = 0; q < NQ; ++q)
#pragma unroll
        for (int j = 0; j < NB / 2; ++j) acc2[q][j] = pk2(0.0f, 0.0f);
#pragma unroll
    for (int t = 0; t < kWin + NB - 1; ++t) {
        float v[NQ];
        load(t, v);
#pragma unroll
        for (int j = 0; j < NB / 2; ++j) {
            const int k = t - 2 * j;
            if (k >= 0 && k <= kWin) {
                const f32x2 w2 = pk2(win.p[k].x, win.p[k].y);
#pragma unroll
                for (int q = 0; q < NQ; ++q) acc2[q][j] = fma2(w2, bc2(v[q]), acc2[q][j]);
            }
        }
    }
}

// The held-out metrics' view of the kernel (ssim_fwd_kernel<true>): the prediction is clamp(rgb + (1 - alpha) bg, 0, 1)
// of the render, formed as loss_grad_kernel forms it, against the unmasked ground truth.  Each block owns the input pixels
// [x0, x0 + 32) x [y0, y0 + 32) of its tile (the last tile of a row / column also the up to 10 pixels after them: together
// every pixel once) and writes, in fixed order, partials[(cam * 3 + ch) * tiles + tile][kEvalPartials] =
//   {sum SSIM map, sum (pred - gt)^2 of channel ch, then for ch == 0 (zeros otherwise) over its pixels with finite ground
//    truth > depth_tol: n, sum |g - d| / g, sum (g - d)^2 / g, sum (g - d)^2, sum (log g - log d)^2, and the counts of
//    max(g / d, d / g) < 1.25, 1.25^2, 1.25^3}
// with d = the depth channel where alpha > 0, else the view's fill value fill[cam] (float bits).  Sums in float64.

struct SsimEval {
    const float4* render;  // [C,H,W,4]
    const float* alphas;   // [C,H,W]
    const float* bg;       // [3]
    GtDepth gt_depth;
    const int* fill;       // [C] the view's maximum rendered depth, as float bits
    float depth_tol;
    double* partials;
};

// grid (tiles_x, tiles_y, C*3); 256 threads.
template <bool EVAL>
__global__ void __launch_bounds__(kSsimThreads) ssim_fwd_kernel(int W, int H, const float* __restrict__ pred /*[C,H,W,3]*/,
                                                                const GtImage gt, const PixelMask mask, const GaussWin win,
                                                                float* __restrict__ dmaps /*[C*3][3][OH][OW]*/, double* __restrict__ stats,
                                                                const SsimEval ev = SsimEval{}) {
    extern __shared__ __align__(16) float ssim_smem[];
    float(*sx)[kSsimIn + 1] = reinterpret_cast<float(*)[kSsimIn + 1]>(ssim_smem);            // [42][43]
    float(*sy)[kSsimIn + 1] = sx + kSsimIn;                                                   // [42][43]
    float(*h)[kSsimIn][kHStride] = reinterpret_cast<float(*)[kSsimIn][kHStride]>(ssim_smem + 2 * kSsimIn * (kSsimIn + 1));  // [5][42][34]
    __shared__ double red[kSsimThreads / 32];
    pdl_enter();
    const int OW = W - kHalo, OH = H - kHalo;
    const int cam = blockIdx.z / 3, ch = blockIdx.z % 3;
    const int ox0 = blockIdx.x * kSsimTile, oy0 = blockIdx.y * kSsimTile;
    const int64_t img = (int64_t)cam * H * W;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int r = warp; r < kSsimIn; r += kSsimThreads / 32) {
        const int y = oy0 + r;
        for (int c = lane; c < kSsimIn; c += 32) {
            const int x = ox0 + c;
            float a = 0.f, b = 0.f;
            if (y < H && x < W) {
                const int64_t pix = img + (int64_t)y * W + x, o = pix * 3 + ch;
                if constexpr (EVAL) {
                    const float4 r4 = ev.render[pix];
                    const float rc = ch == 0 ? r4.x : (ch == 1 ? r4.y : r4.z);
                    a = gt.at(o);
                    b = fminf(fmaxf(rc + (1.0f - ev.alphas[pix]) * ev.bg[ch], 0.0f), 1.0f);
                } else {
                    a = gt.at(o) * mask.at(pix);  // pred already carries the mask (loss_grad_kernel<WRITE_PRED>)
                    b = pred[o];
                }
            }
            sx[r][c] = a;
            sy[r][c] = b;
        }
    }
    __syncthreads();
    double part[kEvalPartials - 1] = {};  // EVAL: this thread's share of the partials after the SSIM sum
    if constexpr (EVAL) {
        // the pixels this block owns (see SsimEval)
        const int tiles_x = gridDim.x, tiles_y = gridDim.y;
        const int nx = (int)blockIdx.x == tiles_x - 1 ? W - ox0 : kSsimTile, ny = (int)blockIdx.y == tiles_y - 1 ? H - oy0 : kSsimTile;
        const float fill = __int_as_float(ev.fill[cam]);
        for (int i = threadIdx.x; i < nx * ny; i += kSsimThreads) {
            const int r = i / nx, c = i % nx;
            const double e = (double)sy[r][c] - (double)sx[r][c];
            part[0] += e * e;
            if (ch != 0) continue;
            const int64_t pix = img + (int64_t)(oy0 + r) * W + ox0 + c;
            const float gf = ev.gt_depth.at(pix);
            if (!(fabsf(gf) <= 3.402823466e38f && gf > ev.depth_tol)) continue;
            const double g = gf, d = ev.alphas[pix] > 0.0f ? ev.render[pix].w : fill;
            const double diff = g - d, lg = log(g) - log(d);
            const double t = fmax(g / d, d / g);
            part[1] += 1.0;
            part[2] += fabs(diff) / g;
            part[3] += diff * diff / g;
            part[4] += diff * diff;
            part[5] += lg * lg;
            part[6] += t < 1.25 ? 1.0 : 0.0;
            part[7] += t < 1.25 * 1.25 ? 1.0 : 0.0;
            part[8] += t < 1.25 * 1.25 * 1.25 ? 1.0 : 0.0;
        }
    }
    // horizontal pass: 42 rows x (32 / kBlkH) column groups = 168 items
    if (threadIdx.x < kSsimIn * (kSsimTile / kBlkH)) {
        const int r = threadIdx.x / (kSsimTile / kBlkH), c0 = (threadIdx.x % (kSsimTile / kBlkH)) * kBlkH;
        f32x2 acc2[5][kBlkH / 2];
        filter_taps<5, kBlkH>(win, acc2, [&](int t, float(&v)[5]) {
            const float a = sx[r][c0 + t], b = sy[r][c0 + t];
            v[0] = a;
            v[1] = b;
            v[2] = a * a;
            v[3] = b * b;
            v[4] = a * b;
        });
#pragma unroll
        for (int q = 0; q < 5; ++q)
#pragma unroll
            for (int j = 0; j < kBlkH / 2; ++j) *reinterpret_cast<f32x2*>(&h[q][r][c0 + 2 * j]) = acc2[q][j];
    }
    __syncthreads();
    // vertical pass: 32 columns x (32 / kBlkV) row groups = 256 items
    float local_f = 0.0f;  // <= 4 maps in [-1, 1] per thread: summed in float, then in double across the CTA / image
    {
        const int tx = threadIdx.x % kSsimTile, y0 = (threadIdx.x / kSsimTile) * kBlkV;
        f32x2 acc2[5][kBlkV / 2];
        filter_taps<5, kBlkV>(win, acc2, [&](int t, float(&v)[5]) {
#pragma unroll
            for (int q = 0; q < 5; ++q) v[q] = h[q][y0 + t][tx];
        });
        const float C1 = 0.01f * 0.01f, C2 = 0.03f * 0.03f;
        const int64_t plane = (int64_t)OH * OW;
        const int ox = ox0 + tx;
#pragma unroll
        for (int o = 0; o < kBlkV; ++o) {
            const int oy = oy0 + y0 + o;
            if (oy < OH && ox < OW) {
                float m[5];
#pragma unroll
                for (int q = 0; q < 5; ++q) m[q] = (o & 1) ? hi2(acc2[q][o / 2]) : lo2(acc2[q][o / 2]);
                const float m1 = m[0], m2 = m[1], e1 = m[2], e2 = m[3], e12 = m[4];
                const float s1 = e1 - m1 * m1, s2 = e2 - m2 * m2, s12 = e12 - m1 * m2;
                const float A1 = 2.f * m1 * m2 + C1, A2 = 2.f * s12 + C2, B1 = m1 * m1 + m2 * m2 + C1, B2 = s1 + s2 + C2;
                // reciprocals by rcp.approx (1 ulp) instead of IEEE divisions (~14 instructions each): far inside the 1e-4 tolerance
                const float rB2 = rcp_approx(B2);
                const float inv = rcp_approx(B1) * rB2;
                const float map = A1 * A2 * inv;
                local_f += map;
                if constexpr (!EVAL) {
                    float* d = dmaps + ((int64_t)blockIdx.z * 3) * plane + (int64_t)oy * OW + ox;
                    d[0] = (2.f * m1 * (A2 - A1) - 2.f * m2 * map * (B2 - B1)) * inv;  // d map / d mu2 (e2, e12 fixed)
                    d[plane] = -map * rB2;                                             // d map / d e2
                    d[2 * plane] = 2.f * A1 * inv;                                     // d map / d e12
                }
            }
        }
    }
    double local = (double)local_f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if constexpr (EVAL) {
        // fixed-order block sums: xor shuffles inside each warp, then the warps in order
        __shared__ double red_p[kSsimThreads / 32][kEvalPartials - 1];
#pragma unroll
        for (int k = 0; k < kEvalPartials - 1; ++k) {
            double v = part[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) red_p[warp][k] = v;
        }
        if (lane == 0) red[warp] = local;
        __syncthreads();
        if (threadIdx.x < kEvalPartials) {
            const int k = threadIdx.x;
            double s = 0;
            for (int i = 0; i < kSsimThreads / 32; ++i) s += k == 0 ? red[i] : red_p[i][k - 1];
            const int64_t tile = (int64_t)blockIdx.y * gridDim.x + blockIdx.x;
            ev.partials[((int64_t)blockIdx.z * gridDim.x * gridDim.y + tile) * kEvalPartials + k] = s;
        }
    } else {
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0;
            for (int i = 0; i < kSsimThreads / 32; ++i) s += red[i];
            atomicAdd(stats + cam * 8 + 5, s);
        }
    }
}

// grid (ceil(W/32), ceil(H/32), C*3): dL/dpred for a 32x32 tile of INPUT pixels
__global__ void __launch_bounds__(kSsimThreads) ssim_bwd_kernel(int W, int H, const float* __restrict__ pred, const GtImage gt, const PixelMask mask,
                                                                const GaussWin win, const float* __restrict__ dmaps, float scale,
                                                                float* __restrict__ v_pred /*[C,H,W,3]*/) {
    extern __shared__ __align__(16) float ssim_smem[];
    float(*sd)[kSsimIn][kSsimIn + 1] = reinterpret_cast<float(*)[kSsimIn][kSsimIn + 1]>(ssim_smem);                           // [3][42][43]
    float(*h)[kSsimIn][kHStride] = reinterpret_cast<float(*)[kSsimIn][kHStride]>(ssim_smem + 3 * kSsimIn * (kSsimIn + 1) + 2);  // [3][42][34], 8-B aligned
    pdl_enter();
    const int OW = W - kHalo, OH = H - kHalo;
    const int cam = blockIdx.z / 3, ch = blockIdx.z % 3;
    const int x0 = blockIdx.x * kSsimTile, y0 = blockIdx.y * kSsimTile;
    const int64_t plane = (int64_t)OH * OW;
    const float* d = dmaps + ((int64_t)blockIdx.z * 3) * plane;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // pixel p gets contributions from q in [p-10, p] (valid coords): load the q tile starting at (y0-10, x0-10)
    for (int r = warp; r < kSsimIn; r += kSsimThreads / 32) {
        const int qy = y0 - kHalo + r;
        for (int c = lane; c < kSsimIn; c += 32) {
            const int qx = x0 - kHalo + c;
            float a = 0.f, b = 0.f, e = 0.f;
            if (qy >= 0 && qy < OH && qx >= 0 && qx < OW) {
                const int64_t o = (int64_t)qy * OW + qx;
                a = d[o];
                b = d[plane + o];
                e = d[2 * plane + o];
            }
            sd[0][r][c] = a;
            sd[1][r][c] = b;
            sd[2][r][c] = e;
        }
    }
    __syncthreads();
    // pixel p = x0 + c receives q = p - 10 + k with weight w[10 - k] = w[k] (the window is symmetric)
    if (threadIdx.x < kSsimIn * (kSsimTile / kBlkH)) {
        const int r = threadIdx.x / (kSsimTile / kBlkH), c0 = (threadIdx.x % (kSsimTile / kBlkH)) * kBlkH;
        f32x2 acc2[3][kBlkH / 2];
        filter_taps<3, kBlkH>(win, acc2, [&](int t, float(&v)[3]) {
            v[0] = sd[0][r][c0 + t];
            v[1] = sd[1][r][c0 + t];
            v[2] = sd[2][r][c0 + t];
        });
#pragma unroll
        for (int q = 0; q < 3; ++q)
#pragma unroll
            for (int j = 0; j < kBlkH / 2; ++j) *reinterpret_cast<f32x2*>(&h[q][r][c0 + 2 * j]) = acc2[q][j];
    }
    __syncthreads();
    {
        const int tx = threadIdx.x % kSsimTile, yb = (threadIdx.x / kSsimTile) * kBlkV;
        f32x2 acc2[3][kBlkV / 2];
        filter_taps<3, kBlkV>(win, acc2, [&](int t, float(&v)[3]) {
            v[0] = h[0][yb + t][tx];
            v[1] = h[1][yb + t][tx];
            v[2] = h[2][yb + t][tx];
        });
        const int x = x0 + tx;
#pragma unroll
        for (int o = 0; o < kBlkV; ++o) {
            const int y = y0 + yb + o;
            if (y < H && x < W) {
                const float a0 = (o & 1) ? hi2(acc2[0][o / 2]) : lo2(acc2[0][o / 2]);
                const float a1 = (o & 1) ? hi2(acc2[1][o / 2]) : lo2(acc2[1][o / 2]);
                const float a2 = (o & 1) ? hi2(acc2[2][o / 2]) : lo2(acc2[2][o / 2]);
                const int64_t pix = ((int64_t)cam * H + y) * W + x, idx = pix * 3 + ch;
                v_pred[idx] = scale * (a0 + 2.f * pred[idx] * a1 + gt.at(idx) * mask.at(pix) * a2);
            }
        }
    }
}

constexpr size_t kSsimFwdSmem = (size_t)(2 * kSsimIn * (kSsimIn + 1) + 5 * kSsimIn * kHStride) * 4;
constexpr size_t kSsimBwdSmem = (size_t)(3 * kSsimIn * (kSsimIn + 1) + 2 + 3 * kSsimIn * kHStride) * 4;

}  // namespace qed

using namespace qed;

// pred (already multiplied by the mask) / gt [C,H,W,3], mask [C,H,W] or NULL; dmaps scratch [C*3*3*(H-10)*(W-10)]; stats[c*8+5] += sum of the SSIM map of camera c;
// v_pred = scale * d(sum map)/d pred.  Internal to qed_loss_fwd_bwd (train.cu), declared there.
int qed_ssim_launch(int C, int W, int H, const float* pred, qed::GtImage gt, qed::PixelMask mask, float* dmaps, double* stats, float scale,
                    float* v_pred, cudaStream_t stream) {
    if (W <= kHalo || H <= kHalo) return QED_ERR_UNSUPPORTED;
    static const GaussWin win = make_window();
    const int OW = W - kHalo, OH = H - kHalo;
    QED_CUDA_TRY(cudaFuncSetAttribute(ssim_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSsimFwdSmem));
    QED_CUDA_TRY(cudaFuncSetAttribute(ssim_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSsimBwdSmem));
    dim3 g1((OW + kSsimTile - 1) / kSsimTile, (OH + kSsimTile - 1) / kSsimTile, C * 3);
    QED_CUDA_TRY(launch_pdl(ssim_fwd_kernel<false>, g1, dim3(kSsimThreads), kSsimFwdSmem, stream, W, H, pred, gt, mask, win, dmaps, stats, SsimEval{}));
    dim3 g2((W + kSsimTile - 1) / kSsimTile, (H + kSsimTile - 1) / kSsimTile, C * 3);
    QED_CUDA_TRY(launch_pdl(ssim_bwd_kernel, g2, dim3(kSsimThreads), kSsimBwdSmem, stream, W, H, pred, gt, mask, win, dmaps, scale, v_pred));
    return QED_OK;
}

// Tiles (blocks per view and channel) of qed_ssim_eval_launch: its partials are [C*3][tiles][kEvalPartials] doubles.
int64_t qed_ssim_eval_tiles(int W, int H) {
    return (int64_t)((W - kHalo + kSsimTile - 1) / kSsimTile) * ((H - kHalo + kSsimTile - 1) / kSsimTile);
}

// The held-out metrics' pass (ssim_fwd_kernel<true>, see SsimEval).  Internal to qed_eval_metrics (metrics.cu), declared there.
int qed_ssim_eval_launch(int C, int W, int H, const float* render, const float* alphas, qed::GtImage gt, qed::GtDepth gt_depth, const float* bg,
                         const int* fill, float depth_tol, double* partials, cudaStream_t stream) {
    if (W <= kHalo || H <= kHalo) return QED_ERR_UNSUPPORTED;
    static const GaussWin win = make_window();
    QED_CUDA_TRY(cudaFuncSetAttribute(ssim_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSsimFwdSmem));
    const SsimEval ev{reinterpret_cast<const float4*>(render), alphas, bg, gt_depth, fill, depth_tol, partials};
    dim3 g((W - kHalo + kSsimTile - 1) / kSsimTile, (H - kHalo + kSsimTile - 1) / kSsimTile, C * 3);
    QED_CUDA_TRY(launch_pdl(ssim_fwd_kernel<true>, g, dim3(kSsimThreads), kSsimFwdSmem, stream, W, H, (const float*)nullptr, gt, PixelMask{nullptr, 0}, win,
                            (float*)nullptr, (double*)nullptr, ev));
    return QED_OK;
}
