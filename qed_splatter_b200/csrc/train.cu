// Loss + loss-gradient fusion (SURVEY.md §8 rows a11-a13) and trainer-side kernels (a14, a16).
//
// qed_loss_fwd_bwd replaces the autograd graph the reference builds at qed_splatter/model.py:295-306
// (background composite, clamp, depth fill with the detached max) and :87-116 (depth-L1 over
// finite & gt>0 pixels times depth_lambda) plus the L1 term of splatfacto's RGB loss (model.py:83-85).
// Every camera is one reference step: its depth term is normalised by ITS n_valid, its depth fill uses
// ITS max; the batch loss is the mean over cameras.
// qed_adam_arena replaces the 6 torch Adam groups of qed_splatter/config.py:44-68 with one launch over a
// flat arena; qed_strategy_update is gsplat DefaultStrategy._update_state on the `info` of model.py:267,289-292.
#include "common.cuh"

namespace qed {

constexpr int kLossThreads = 256;
constexpr int kLossUnroll = 4;

__device__ __forceinline__ float signf(float x) { return (x > 0.0f) ? 1.0f : ((x < 0.0f) ? -1.0f : 0.0f); }
__device__ __forceinline__ bool finitef(float x) { return fabsf(x) <= 3.402823466e38f; }

// pass 1 (24 B/pixel): per camera max of the depth channel (the fill value of model.py:304-306) and the number of
// pixels the depth loss averages over (model.py:101-105).  The depth channel is >= 0, so the integer order of the
// float bits is the float order and atomicMax on the bits works.  stats[2] = valid pixels with alpha > 0,
// stats[6] = pixels with alpha == 0 whose ground truth is usable (valid iff the fill value is finite).
__global__ void __launch_bounds__(kLossThreads) loss_stats_kernel(int64_t HW, const float4* __restrict__ render, const float* __restrict__ alphas,
                                                                 const GtDepth gt_depth, const PixelMask mask, double* __restrict__ stats) {
    __shared__ float s_max[kLossThreads / 32];
    __shared__ int s_na[kLossThreads / 32], s_nb[kLossThreads / 32];
    pdl_enter();
    const int cam = blockIdx.y;
    float maxd = 0.0f;
    int na = 0, nb = 0;
    const int64_t base = (int64_t)blockIdx.x * (kLossThreads * kLossUnroll) + threadIdx.x;
    float d[kLossUnroll], a[kLossUnroll], gd[kLossUnroll], mk[kLossUnroll];
#pragma unroll
    for (int u = 0; u < kLossUnroll; ++u) {  // all loads first: kLossUnroll independent requests in flight per thread
        const int64_t i = base + (int64_t)u * kLossThreads;
        const bool in = i < HW;
        const int64_t pix = cam * HW + (in ? i : 0);
        d[u] = in ? render[pix].w : 0.0f;
        a[u] = in ? alphas[pix] : 1.0f;
        gd[u] = in ? gt_depth.at(pix) : 0.0f;
        mk[u] = in ? mask.at(pix) : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < kLossUnroll; ++u) {
        maxd = fmaxf(maxd, d[u]);  // the fill value is the maximum of the UNMASKED rendered depth (model.py:304-306 run before the loss)
        const float gm = gd[u] * mk[u];  // model.py:96-97: both sides are multiplied by the mask before the validity test
        const bool gt_ok = finitef(gm) && gm > 0.0f;
        if (a[u] > 0.0f) na += (gt_ok && finitef(d[u] * mk[u])) ? 1 : 0;
        else nb += gt_ok ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        maxd = fmaxf(maxd, __shfl_xor_sync(0xffffffffu, maxd, o));
        na += __shfl_xor_sync(0xffffffffu, na, o);
        nb += __shfl_xor_sync(0xffffffffu, nb, o);
    }
    if ((threadIdx.x & 31) == 0) {
        s_max[threadIdx.x >> 5] = maxd;
        s_na[threadIdx.x >> 5] = na;
        s_nb[threadIdx.x >> 5] = nb;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kLossThreads / 32; ++w) {
            maxd = fmaxf(maxd, s_max[w]);
            na += s_na[w];
            nb += s_nb[w];
        }
        atomicMax(reinterpret_cast<int*>(stats + cam * 8 + 3), __float_as_int(maxd));
        if (na) atomicAdd(stats + cam * 8 + 2, (double)na);
        if (nb) atomicAdd(stats + cam * 8 + 6, (double)nb);
    }
}

__device__ __forceinline__ double n_valid_of(const double* s, float maxd) { return s[2] + (finitef(maxd) ? s[6] : 0.0); }

// ---- splatfacto's bilateral grid (nerfstudio lib_bilagrid `slice`), applied to the clamped rgb of training views ----
// grids[G,12,L,Y,X]: per training image a 3x4 affine colour matrix A[i][j] = ch[4i+j] on an X x Y x L lattice.  A pixel
// (row h, column w) looks up x = w/(W-1), y = h/(H-1), z = BT.601 gray of its colour, as grid_sample(align_corners=True,
// padding_mode="border") does: g = coordinate * (n-1), clamped to [0, n-1]; trilinear over the 8 neighbouring cells.
constexpr int kBilagridMaxL = 16;
constexpr int kBilagridMaxXY = 1024;

struct BilagridArgs {
    const float* grids;     // [G,12,L,Y,X]
    const int32_t* ids;     // [C] grid of each view
    int num_grids, W, H, X, Y, L;
    float4* rec_c;          // [C*HW] per pixel {c0, c1, c2, gz} (workspace; written by the gradient pass)
    float4* rec_v;          // [C*HW] per pixel {d loss / d out (3), 0}
};

// lattice coordinate of pixel index p of an axis of n_px pixels on an axis of n cells: cell i0 in [0, n-2] and weight f
// of cell i0 + 1 (f = 1 on the last cell, which grid_sample reaches with weight 1 as well)
__device__ __forceinline__ void bilagrid_axis(int p, int n_px, int n, int& i0, float& f) {
    const float x = n_px > 1 ? (float)p / (float)(n_px - 1) : 0.0f;
    const float g = fminf(fmaxf(x * (float)(n - 1), 0.0f), (float)(n - 1));
    i0 = min((int)floorf(g), n - 2);
    f = g - (float)i0;
}

__device__ __forceinline__ float bilagrid_gz(float c0, float c1, float c2, int L, bool& inside) {
    const float gz = (0.299f * c0 + 0.587f * c1 + 0.114f * c2) * (float)(L - 1);
    inside = gz >= 0.0f && gz <= (float)(L - 1);  // grid_sample's border padding: no gradient through a clamped coordinate
    return fminf(fmaxf(gz, 0.0f), (float)(L - 1));
}

// A[12] (trilinear) at pixel (h, w) with guidance gz of the view's grid g (NULL: NaN, an invalid id), and
// dout[3] = d out_i / d gz for the colour c
__device__ __forceinline__ void bilagrid_sample(const float* __restrict__ g, int X, int Y, int L, int h, int w, int H, int W, float gz,
                                                float c0, float c1, float c2, float A[12], float dout[3]) {
    int x0, y0;
    float fx, fy;
    bilagrid_axis(w, W, X, x0, fx);
    bilagrid_axis(h, H, Y, y0, fy);
    const int z0 = min((int)floorf(gz), L - 2);
    const float fz = gz - (float)z0;
    const int64_t sz = (int64_t)X * Y, sc = sz * L;
    const float wxy[4] = {(1.0f - fx) * (1.0f - fy), fx * (1.0f - fy), (1.0f - fx) * fy, fx * fy};
    const int64_t oxy[4] = {(int64_t)y0 * X + x0, (int64_t)y0 * X + x0 + 1, (int64_t)(y0 + 1) * X + x0, (int64_t)(y0 + 1) * X + x0 + 1};
#pragma unroll
    for (int ch = 0; ch < 12; ++ch) {
        float a = 0.0f, d = 0.0f;
        if (g) {
            const float* gc = g + ch * sc + (int64_t)z0 * sz;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float lo = __ldg(gc + oxy[k]), hi = __ldg(gc + sz + oxy[k]);
                a += wxy[k] * ((1.0f - fz) * lo + fz * hi);
                d += wxy[k] * (hi - lo);
            }
        } else {
            a = d = __int_as_float(0x7fffffff);
        }
        A[ch] = a;
        const float cj = (ch & 3) == 0 ? c0 : ((ch & 3) == 1 ? c1 : ((ch & 3) == 2 ? c2 : 1.0f));
        if ((ch & 3) == 0) dout[ch >> 2] = d * cj;
        else dout[ch >> 2] += d * cj;
    }
}

// pass 2 (68 B/pixel): per-pixel loss terms and their gradient w.r.t. the compositor outputs.
//   WRITE_PRED : only write the clamped rgb image (input of the SSIM kernels), no sums, no gradients
//   otherwise  : loss sums + gradients (v_rgb_extra = gradient of the SSIM term w.r.t. the clamped rgb, or NULL)
//   BILAGRID   : the loss sees the clamped rgb after the view's bilateral grid; the gradient pass chains through the slice
//                and leaves per-pixel records for bilagrid_grad_kernel
template <bool WRITE_PRED, bool BILAGRID = false>
__global__ void __launch_bounds__(kLossThreads) loss_grad_kernel(int64_t HW, int C, const float4* __restrict__ render, const float* __restrict__ alphas,
                                                                const GtImage gt_rgb, const GtDepth gt_depth, const PixelMask mask,
                                                                const float* __restrict__ bg, float rgb_weight, float depth_lambda, float grad_scale,
                                                                double* __restrict__ stats, float4* __restrict__ v_render, float* __restrict__ v_alphas,
                                                                float* __restrict__ pred_rgb, const float* __restrict__ v_rgb_extra,
                                                                const BilagridArgs bla = BilagridArgs{}) {
    pdl_enter();
    const int cam = blockIdx.y;
    const float maxd = __int_as_float(*reinterpret_cast<const int*>(stats + cam * 8 + 3));
    const float b0 = bg[0], b1 = bg[1], b2 = bg[2];
    double s_rgb = 0.0, s_d = 0.0;
    const double nv = n_valid_of(stats + cam * 8, maxd);
    const float inv_nvalid = nv > 0.0 ? (float)(1.0 / nv) : 0.0f;
    const float g_rgb = rgb_weight * grad_scale / ((float)C * (float)HW * 3.0f);
    const float g_d = depth_lambda * grad_scale * inv_nvalid / (float)C;
#pragma unroll
    for (int u = 0; u < kLossUnroll; ++u) {
        const int64_t i = (int64_t)blockIdx.x * (kLossThreads * kLossUnroll) + (int64_t)u * kLossThreads + threadIdx.x;
        if (i >= HW) continue;
        const int64_t pix = cam * HW + i;
        const float4 r = render[pix];
        const float a = alphas[pix];
        const float om = 1.0f - a;
        const float pre0 = r.x + om * b0, pre1 = r.y + om * b1, pre2 = r.z + om * b2;
        const float c0 = fminf(fmaxf(pre0, 0.0f), 1.0f), c1 = fminf(fmaxf(pre1, 0.0f), 1.0f), c2 = fminf(fmaxf(pre2, 0.0f), 1.0f);
        const float mk = mask.at(pix);  // 1 without a mask: every product below is then exact
        float o0 = c0, o1 = c1, o2 = c2;  // the colour the loss sees
        float A[BILAGRID ? 12 : 1], dout[3], gz = 0.0f;
        bool z_in = false;
        if constexpr (BILAGRID) {
            const int gid = bla.ids[cam];
            const float* g = (gid >= 0 && gid < bla.num_grids) ? bla.grids + (int64_t)gid * 12 * bla.L * bla.Y * bla.X : nullptr;
            gz = bilagrid_gz(c0, c1, c2, bla.L, z_in);
            bilagrid_sample(g, bla.X, bla.Y, bla.L, (int)(i / bla.W), (int)(i % bla.W), bla.H, bla.W, gz, c0, c1, c2, A, dout);
            o0 = A[0] * c0 + A[1] * c1 + A[2] * c2 + A[3];
            o1 = A[4] * c0 + A[5] * c1 + A[6] * c2 + A[7];
            o2 = A[8] * c0 + A[9] * c1 + A[10] * c2 + A[11];
        }
        if (WRITE_PRED) {  // splatfacto multiplies prediction and ground truth by the mask before L1 and SSIM
            pred_rgb[pix * 3 + 0] = o0 * mk;
            pred_rgb[pix * 3 + 1] = o1 * mk;
            pred_rgb[pix * 3 + 2] = o2 * mk;
            continue;
        }
        const float e0 = __fmul_rn(o0, mk) - __fmul_rn(gt_rgb.at(pix * 3 + 0), mk), e1 = __fmul_rn(o1, mk) - __fmul_rn(gt_rgb.at(pix * 3 + 1), mk),
                    e2 = __fmul_rn(o2, mk) - __fmul_rn(gt_rgb.at(pix * 3 + 2), mk);
        const float gd = __fmul_rn(gt_depth.at(pix), mk);              // model.py:96-97
        const float d = __fmul_rn((a > 0.0f) ? r.w : maxd, mk);
        const bool valid = finitef(d) && finitef(gd) && (gd > 0.0f);
        s_rgb += (double)(fabsf(e0) + fabsf(e1) + fabsf(e2));
        if (valid) s_d += (double)fabsf(d - gd);
        float x0 = 0.f, x1 = 0.f, x2 = 0.f;  // gradient of the SSIM term w.r.t. the clamped rgb
        if (v_rgb_extra) {  // gradient w.r.t. the masked prediction -> chain rule through the mask product
            x0 = v_rgb_extra[pix * 3 + 0] * mk;
            x1 = v_rgb_extra[pix * 3 + 1] * mk;
            x2 = v_rgb_extra[pix * 3 + 2] * mk;
        }
        const float gm_rgb = g_rgb * mk, gm_d = g_d * mk;
        float4 v;
        if constexpr (BILAGRID) {
            // d loss / d out, then through out_i = sum_j A[i][j] c_j + A[i][3] (A depends on c through gz) to c
            const float u0 = gm_rgb * signf(e0) + x0, u1 = gm_rgb * signf(e1) + x1, u2 = gm_rgb * signf(e2) + x2;
            bla.rec_c[pix] = make_float4(c0, c1, c2, gz);
            bla.rec_v[pix] = make_float4(u0, u1, u2, 0.0f);
            float vz = 0.0f;
            if (z_in) vz = (u0 * dout[0] + u1 * dout[1] + u2 * dout[2]) * (float)(bla.L - 1);
            const float w0 = u0 * A[0] + u1 * A[4] + u2 * A[8] + 0.299f * vz, w1 = u0 * A[1] + u1 * A[5] + u2 * A[9] + 0.587f * vz,
                        w2 = u0 * A[2] + u1 * A[6] + u2 * A[10] + 0.114f * vz;
            v.x = (pre0 >= 0.0f && pre0 <= 1.0f) ? w0 : 0.0f;
            v.y = (pre1 >= 0.0f && pre1 <= 1.0f) ? w1 : 0.0f;
            v.z = (pre2 >= 0.0f && pre2 <= 1.0f) ? w2 : 0.0f;
        } else {
            v.x = (pre0 >= 0.0f && pre0 <= 1.0f) ? gm_rgb * signf(e0) + x0 : 0.0f;
            v.y = (pre1 >= 0.0f && pre1 <= 1.0f) ? gm_rgb * signf(e1) + x1 : 0.0f;
            v.z = (pre2 >= 0.0f && pre2 <= 1.0f) ? gm_rgb * signf(e2) + x2 : 0.0f;
        }
        v.w = (valid && a > 0.0f) ? gm_d * signf(d - gd) : 0.0f;
        v_render[pix] = v;
        v_alphas[pix] = -(v.x * b0 + v.y * b1 + v.z * b2);
    }
    if (!WRITE_PRED) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s_rgb += __shfl_xor_sync(0xffffffffu, s_rgb, o);
            s_d += __shfl_xor_sync(0xffffffffu, s_d, o);
        }
        __shared__ double s_a[kLossThreads / 32], s_b[kLossThreads / 32];
        if ((threadIdx.x & 31) == 0) {
            s_a[threadIdx.x >> 5] = s_rgb;
            s_b[threadIdx.x >> 5] = s_d;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < kLossThreads / 32; ++w) {
                s_rgb += s_a[w];
                s_d += s_b[w];
            }
            atomicAdd(stats + cam * 8 + 0, s_rgb);
            atomicAdd(stats + cam * 8 + 1, s_d);
        }
    }
}

__global__ void loss_finalize_kernel(int C, int64_t HW, float rgb_weight, float depth_lambda, float ssim_lambda, double ssim_count,
                                     double* __restrict__ stats, float* __restrict__ loss) {
    pdl_enter();
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double lr = 0.0, ld = 0.0, ls = 0.0;
    for (int c = 0; c < C; ++c) {
        double* s = stats + c * 8;
        lr += s[0] / ((double)HW * 3.0);
        if (ssim_lambda > 0.0f) ls += 1.0 - s[5] / ssim_count;
        const float maxd = __int_as_float(*reinterpret_cast<const int*>(s + 3));
        const double nv = n_valid_of(s, maxd);
        ld += nv > 0.0 ? s[1] / nv : 0.0;
        s[2] = nv;
        s[4] = (double)maxd;
    }
    lr = rgb_weight * lr / C + ssim_lambda * ls / C;
    ld = depth_lambda * ld / C;
    loss[0] = (float)(lr + ld);
    loss[1] = (float)lr;
    loss[2] = (float)ld;
}

// Bilateral-grid gradient, gathered: one block per (lattice column (ix, iy), ROWS output rows of A starting at blockIdx.y *
// ROWS, view).  It visits the pixels whose x / y cell touches the column, in a fixed order (warps over consecutive columns of
// an image row), and keeps sum_pixels w * d loss / d out_i * [c, 1] for every level of the column in registers; then a
// fixed-order block reduction (xor shuffles, warps in order) writes the ROWS x 4 x L values.  No atomics: the same inputs
// give the same bits.  v_grid_rows[C,12,L,Y,X] is overwritten.
constexpr int kBilagridThreads = 256;

template <int LM, int ROWS>
__global__ void __launch_bounds__(kBilagridThreads) bilagrid_grad_kernel(int64_t HW, const BilagridArgs bla, float* __restrict__ v_rows) {
    __shared__ float s_part[kBilagridThreads / 32][ROWS * 4 * LM];
    pdl_enter();
    const int X = bla.X, Y = bla.Y, L = bla.L, W = bla.W, H = bla.H;
    const int ix = blockIdx.x % X, iy = blockIdx.x / X, row0 = blockIdx.y * ROWS, cam = blockIdx.z;
    // pixels whose cell is ix-1 or ix (resp. iy-1 or iy), with one pixel of slack each side; the weights decide exactly
    auto span = [](int i, int n, int n_px, int& lo, int& hi) {
        const double s = n_px > 1 ? (double)(n_px - 1) / (double)(n - 1) : 0.0;
        lo = max(0, (int)floor((i - 1) * s) - 1);
        hi = min(n_px - 1, (int)ceil((i + 1) * s) + 1);
    };
    int w_lo, w_hi, h_lo, h_hi;
    span(ix, X, W, w_lo, w_hi);
    span(iy, Y, H, h_lo, h_hi);
    float acc[ROWS][LM][4];
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
        for (int l = 0; l < LM; ++l)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[r][l][j] = 0.0f;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int w = w_lo + lane; w <= w_hi; w += 32) {
        int x0;
        float fx;
        bilagrid_axis(w, W, X, x0, fx);
        const float wx = x0 == ix ? 1.0f - fx : (x0 + 1 == ix ? fx : 0.0f);
        if (wx == 0.0f) continue;
        for (int h = h_lo + warp; h <= h_hi; h += kBilagridThreads / 32) {
            int y0;
            float fy;
            bilagrid_axis(h, H, Y, y0, fy);
            const float wy = y0 == iy ? 1.0f - fy : (y0 + 1 == iy ? fy : 0.0f);
            if (wy == 0.0f) continue;
            const int64_t pix = (int64_t)cam * HW + (int64_t)h * W + w;
            const float4 c = bla.rec_c[pix];
            const float4 u = bla.rec_v[pix];
            const int z0 = min((int)floorf(c.w), L - 2);
            const float fz = c.w - (float)z0, wxy = wx * wy;
#pragma unroll
            for (int r = 0; r < ROWS; ++r) {
                const int row = row0 + r;
                const float val = wxy * (row == 0 ? u.x : (row == 1 ? u.y : u.z));
                const float a0 = (1.0f - fz) * val, a1 = fz * val;
#pragma unroll
                for (int l = 0; l < LM; ++l) {
                    const float wl = l == z0 ? a0 : (l == z0 + 1 ? a1 : 0.0f);
                    acc[r][l][0] += wl * c.x;
                    acc[r][l][1] += wl * c.y;
                    acc[r][l][2] += wl * c.z;
                    acc[r][l][3] += wl;
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
        for (int l = 0; l < LM; ++l)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float a = acc[r][l][j];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
                if (lane == 0) s_part[warp][(r * LM + l) * 4 + j] = a;
            }
    __syncthreads();
    for (int t = threadIdx.x; t < ROWS * 4 * L; t += kBilagridThreads) {
        const int r = t / (4 * L), l = (t >> 2) % L, j = t & 3, k = (r * LM + l) * 4 + j;
        float a = s_part[0][k];
        for (int wp = 1; wp < kBilagridThreads / 32; ++wp) a += s_part[wp][k];
        v_rows[(((int64_t)cam * 12 + (row0 + r) * 4 + j) * L + l) * Y * X + (int64_t)iy * X + ix] = a;
    }
}

// ------------------------------------------------------------------------------------------------
// Two float4 (or, in the scalar tail/unaligned variant, one float) per thread: 8 x LDG.128 issued before anything
// depends on them, streaming loads/stores (read once, written once: keep them out of L2's way), 3 x 2 STG.128.
// 28 B/parameter of pure HBM traffic.
__device__ __forceinline__ float4 ld_stream4(const float* p) { return __ldcs(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st_stream4(float* p, float4 v) { __stcs(reinterpret_cast<float4*>(p), v); }

template <bool VEC4>
__global__ void __launch_bounds__(256) adam_arena_kernel(int64_t n, float* __restrict__ param, const float* __restrict__ grad, float* __restrict__ m,
                                                         float* __restrict__ v, int G, const int64_t* __restrict__ group_ends,
                                                         const float* __restrict__ lr_by_group, const float* __restrict__ lr_alt_by_group,
                                                         const int32_t* __restrict__ group_period, const int32_t* __restrict__ group_split, float beta1,
                                                         float beta2, float eps, float inv_bias1, float inv_bias2_sqrt) {
    __shared__ int64_t s_ends[16];
    __shared__ float s_lr[16], s_lr_alt[16];
    __shared__ int s_period[16], s_split[16];
    pdl_enter();
    if (threadIdx.x < G) {
        s_ends[threadIdx.x] = group_ends[threadIdx.x];
        s_lr[threadIdx.x] = lr_by_group[threadIdx.x];
        s_lr_alt[threadIdx.x] = lr_alt_by_group ? lr_alt_by_group[threadIdx.x] : lr_by_group[threadIdx.x];
        s_period[threadIdx.x] = group_period ? group_period[threadIdx.x] : 0;
        s_split[threadIdx.x] = group_split ? group_split[threadIdx.x] : 0;
    }
    __syncthreads();
    constexpr int W = VEC4 ? 4 : 1;   // consecutive parameters per chunk
    constexpr int U = VEC4 ? 2 : 1;   // chunks per thread, blockDim apart (coalesced)
    const int64_t base = ((int64_t)blockIdx.x * (blockDim.x * U) + threadIdx.x) * W;
    float p[U][W], g[U][W], mi[U][W], vi[U][W];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int64_t i0 = base + (int64_t)u * blockDim.x * W;
        if (i0 >= n) continue;
        if (VEC4) {
            const float4 P = ld_stream4(param + i0), Gd = ld_stream4(grad + i0), M = ld_stream4(m + i0), V = ld_stream4(v + i0);
            p[u][0] = P.x; p[u][W > 1 ? 1 : 0] = P.y; p[u][W > 1 ? 2 : 0] = P.z; p[u][W > 1 ? 3 : 0] = P.w;
            g[u][0] = Gd.x; g[u][W > 1 ? 1 : 0] = Gd.y; g[u][W > 1 ? 2 : 0] = Gd.z; g[u][W > 1 ? 3 : 0] = Gd.w;
            mi[u][0] = M.x; mi[u][W > 1 ? 1 : 0] = M.y; mi[u][W > 1 ? 2 : 0] = M.z; mi[u][W > 1 ? 3 : 0] = M.w;
            vi[u][0] = V.x; vi[u][W > 1 ? 1 : 0] = V.y; vi[u][W > 1 ? 2 : 0] = V.z; vi[u][W > 1 ? 3 : 0] = V.w;
        } else {
            p[u][0] = param[i0];
            g[u][0] = grad[i0];
            mi[u][0] = m[i0];
            vi[u][0] = v[i0];
        }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int64_t i0 = base + (int64_t)u * blockDim.x * W;
        if (i0 >= n) continue;
        // group and position inside its lr period, once per chunk (groups are 16-B aligned, but a period need not be:
        // the position is advanced per element)
        int gi = 0;
        while (gi < G - 1 && i0 >= s_ends[gi]) ++gi;
        int period = s_period[gi], pos = 0;
        if (period > 0) pos = (int)((uint64_t)(i0 - (gi > 0 ? s_ends[gi - 1] : 0)) % (uint32_t)period);
#pragma unroll
        for (int k = 0; k < W; ++k) {
            if (W > 1 && i0 + k >= s_ends[gi] && gi < G - 1) {  // chunk straddles a group boundary (unaligned callers only)
                ++gi;
                period = s_period[gi];
                pos = 0;
            }
            const float lr = (period > 0 && pos >= s_split[gi]) ? s_lr_alt[gi] : s_lr[gi];
            if (period > 0 && ++pos == period) pos = 0;
            mi[u][k] = beta1 * mi[u][k] + (1.0f - beta1) * g[u][k];
            vi[u][k] = beta2 * vi[u][k] + (1.0f - beta2) * g[u][k] * g[u][k];
            const float denom = sqrtf(vi[u][k]) * inv_bias2_sqrt + eps;
            p[u][k] -= (lr * inv_bias1) * (mi[u][k] / denom);
        }
        if (VEC4) {
            st_stream4(param + i0, make_float4(p[u][0], p[u][W > 1 ? 1 : 0], p[u][W > 1 ? 2 : 0], p[u][W > 1 ? 3 : 0]));
            st_stream4(m + i0, make_float4(mi[u][0], mi[u][W > 1 ? 1 : 0], mi[u][W > 1 ? 2 : 0], mi[u][W > 1 ? 3 : 0]));
            st_stream4(v + i0, make_float4(vi[u][0], vi[u][W > 1 ? 1 : 0], vi[u][W > 1 ? 2 : 0], vi[u][W > 1 ? 3 : 0]));
        } else {
            param[i0] = p[u][0];
            m[i0] = mi[u][0];
            v[i0] = vi[u][0];
        }
    }
}

__global__ void strategy_update_kernel(int C, int N, const float4* __restrict__ packed, int use_absgrad, const int32_t* __restrict__ radii,
                                       float sx, float sy, float inv_max_wh, float* __restrict__ grad2d, float* __restrict__ count,
                                       float* __restrict__ radii_max) {
    pdl_enter();
    int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float g = 0.0f, cnt = 0.0f, rm = radii_max ? radii_max[n] : 0.0f;
    for (int c = 0; c < C; ++c) {
        const int64_t idx = (int64_t)c * N + n;
        const int r = radii[idx];
        if (r > 0) {
            const float4 r0 = packed[idx * 3];
            const float gx = (use_absgrad ? r0.z : r0.x) * sx, gy = (use_absgrad ? r0.w : r0.y) * sy;
            g += sqrtf(gx * gx + gy * gy);
            cnt += 1.0f;
            rm = fmaxf(rm, (float)r * inv_max_wh);
        }
    }
    if (cnt > 0.0f) {
        grad2d[n] += g;
        count[n] += cnt;
        if (radii_max) radii_max[n] = rm;
    }
}

}  // namespace qed

using namespace qed;

int qed_ssim_launch(int C, int W, int H, const float* pred, qed::GtImage gt, qed::PixelMask mask, float* dmaps, double* stats, float scale,
                    float* v_pred, cudaStream_t stream);  // ssim.cu

extern "C" size_t qed_loss_workspace_bytes(int C, int width, int height, float ssim_lambda) {
    if (!(ssim_lambda > 0.0f) || C <= 0) return 0;
    const size_t px = (size_t)C * width * height;
    return px * 3 * 4 /* clamped rgb */ + px * 9 * 4 /* derivative maps (upper bound) */ + px * 3 * 4 /* v_ssim */;
}

// qed_loss_fwd_bwd, and with `bla` the same loss on the bilateral-grid-corrected colour.  The workspace of the grid variant
// starts with its 32 B/pixel records; the SSIM buffers follow.
template <bool BILAGRID>
static int loss_fwd_bwd(int C, int width, int height, const float* render, const float* alphas, const void* gt_rgb_, int gt_rgb_is_u8,
                        const void* gt_depth_, int gt_depth_is_u16, double depth_unit_scale, const void* mask_, int mask_is_u8, const float* bg,
                        float rgb_weight, float depth_lambda, float ssim_lambda, float grad_scale, double* stats_dev, float* loss_dev,
                        float* v_render, float* v_alphas, BilagridArgs bla, float* v_grid_rows, void* workspace, size_t workspace_bytes,
                        cudaStream_t stream) {
    if (C <= 0 || width <= 0 || height <= 0) return QED_ERR_BAD_ARG;
    if (!render || !alphas || !gt_rgb_ || !gt_depth_ || !bg || !stats_dev || !loss_dev || !v_render || !v_alphas) return QED_ERR_BAD_ARG;
    const GtImage gt_rgb{gt_rgb_, gt_rgb_is_u8 ? 1 : 0};
    const PixelMask mask{mask_, mask_is_u8 ? 1 : 0};
    const GtDepth gt_depth{gt_depth_, gt_depth_is_u16 ? 1 : 0, depth_unit_scale};
    if (C > 21845) return QED_ERR_UNSUPPORTED;
    const bool use_ssim = ssim_lambda > 0.0f;
    const int64_t HW = (int64_t)width * height;
    const size_t px = (size_t)C * HW;
    const size_t rec_bytes = BILAGRID ? px * 2 * sizeof(float4) : 0;
    if (use_ssim || BILAGRID) {
        if (!workspace) return QED_ERR_BAD_ARG;
        if (workspace_bytes < rec_bytes + qed_loss_workspace_bytes(C, width, height, ssim_lambda)) return QED_ERR_WORKSPACE;
    }
    if (use_ssim && (width <= 10 || height <= 10)) return QED_ERR_UNSUPPORTED;
    if (BILAGRID) {
        bla.rec_c = reinterpret_cast<float4*>(workspace);
        bla.rec_v = bla.rec_c + px;
        workspace = reinterpret_cast<char*>(workspace) + rec_bytes;
    }
    float* pred_rgb = use_ssim ? reinterpret_cast<float*>(workspace) : nullptr;
    float* dmaps = use_ssim ? pred_rgb + px * 3 : nullptr;
    float* v_ssim = use_ssim ? dmaps + px * 9 : nullptr;
    QED_CUDA_TRY(cudaMemsetAsync(stats_dev, 0, (size_t)C * 8 * sizeof(double), stream));
    const int bx = (int)((HW + kLossThreads * kLossUnroll - 1) / (kLossThreads * kLossUnroll));
    dim3 grid(bx, C);
    QED_CUDA_TRY(launch_pdl(loss_stats_kernel, grid, dim3(kLossThreads), 0, stream, HW, reinterpret_cast<const float4*>(render), alphas, gt_depth, mask,
                            stats_dev));
    const double ssim_count = (double)(width - 10) * (double)(height - 10) * 3.0;
    if (use_ssim) {
        QED_CUDA_TRY(launch_pdl(loss_grad_kernel<true, BILAGRID>, grid, dim3(kLossThreads), 0, stream, HW, C, reinterpret_cast<const float4*>(render), alphas,
                                gt_rgb, gt_depth, mask, bg, rgb_weight, depth_lambda, grad_scale, stats_dev, (float4*)nullptr, (float*)nullptr, pred_rgb,
                                (const float*)nullptr, bla));
        // loss term = ssim_lambda * (1 - mean(map)) per camera, mean over cameras
        const float scale = -ssim_lambda * grad_scale / ((float)C * (float)ssim_count);
        int rc = qed_ssim_launch(C, width, height, pred_rgb, gt_rgb, mask, dmaps, stats_dev, scale, v_ssim, stream);
        if (rc != QED_OK) return rc;
    }
    QED_CUDA_TRY(launch_pdl(loss_grad_kernel<false, BILAGRID>, grid, dim3(kLossThreads), 0, stream, HW, C, reinterpret_cast<const float4*>(render), alphas,
                            gt_rgb, gt_depth, mask, bg, rgb_weight, depth_lambda, grad_scale, stats_dev, reinterpret_cast<float4*>(v_render), v_alphas,
                            (float*)nullptr, (const float*)v_ssim, bla));
    if (BILAGRID) {
        // all three output rows per block while their L x 12 sums fit in registers, one row per block above 8 levels
        if (bla.L <= 8)
            QED_CUDA_TRY(launch_pdl(bilagrid_grad_kernel<8, 3>, dim3((unsigned)(bla.X * bla.Y), 1, (unsigned)C), dim3(kBilagridThreads), 0, stream, HW,
                                    (const BilagridArgs)bla, v_grid_rows));
        else
            QED_CUDA_TRY(launch_pdl(bilagrid_grad_kernel<kBilagridMaxL, 1>, dim3((unsigned)(bla.X * bla.Y), 3, (unsigned)C), dim3(kBilagridThreads), 0,
                                    stream, HW, (const BilagridArgs)bla, v_grid_rows));
    }
    QED_CUDA_TRY(launch_pdl(loss_finalize_kernel, dim3(1), dim3(32), 0, stream, C, HW, rgb_weight, depth_lambda, use_ssim ? ssim_lambda : 0.0f, ssim_count,
                            stats_dev, loss_dev));
    return QED_OK;
}

extern "C" int qed_loss_fwd_bwd(int C, int width, int height, const float* render, const float* alphas,
                                const void* gt_rgb_, int gt_rgb_is_u8, const void* gt_depth_, int gt_depth_is_u16, double depth_unit_scale,
                                const void* mask_, int mask_is_u8, const float* bg, float rgb_weight,
                                float depth_lambda, float ssim_lambda, float grad_scale, double* stats_dev, float* loss_dev,
                                float* v_render, float* v_alphas, void* workspace, size_t workspace_bytes, qed_stream_t stream_) {
    return loss_fwd_bwd<false>(C, width, height, render, alphas, gt_rgb_, gt_rgb_is_u8, gt_depth_, gt_depth_is_u16, depth_unit_scale, mask_, mask_is_u8, bg,
                               rgb_weight, depth_lambda, ssim_lambda, grad_scale, stats_dev, loss_dev, v_render, v_alphas, BilagridArgs{}, nullptr,
                               workspace, workspace_bytes, (cudaStream_t)stream_);
}

extern "C" size_t qed_loss_bilagrid_workspace_bytes(int C, int width, int height, float ssim_lambda) {
    if (C <= 0 || width <= 0 || height <= 0) return 0;
    return (size_t)C * width * height * 2 * sizeof(float4) + qed_loss_workspace_bytes(C, width, height, ssim_lambda);
}

extern "C" int qed_loss_fwd_bwd_bilagrid(int C, int width, int height, const float* render, const float* alphas,
                                         const void* gt_rgb, int gt_rgb_is_u8, const void* gt_depth, int gt_depth_is_u16, double depth_unit_scale,
                                         const void* mask, int mask_is_u8, const float* bg, float rgb_weight,
                                         float depth_lambda, float ssim_lambda, float grad_scale, double* stats_dev, float* loss_dev,
                                         float* v_render, float* v_alphas, const float* grids, const int32_t* grid_ids, int num_grids,
                                         int grid_X, int grid_Y, int grid_L, float* v_grid_rows, void* workspace, size_t workspace_bytes,
                                         qed_stream_t stream_) {
    if (!grids || !grid_ids || !v_grid_rows || num_grids <= 0) return QED_ERR_BAD_ARG;
    if (grid_X < 2 || grid_Y < 2 || grid_L < 2 || grid_X > kBilagridMaxXY || grid_Y > kBilagridMaxXY || grid_L > kBilagridMaxL) return QED_ERR_UNSUPPORTED;
    if ((int64_t)grid_X * grid_Y * grid_L * 12 * num_grids > 0x7fffffffLL) return QED_ERR_UNSUPPORTED;
    if (C > 65535) return QED_ERR_UNSUPPORTED;
    BilagridArgs bla{grids, grid_ids, num_grids, width, height, grid_X, grid_Y, grid_L, nullptr, nullptr};
    return loss_fwd_bwd<true>(C, width, height, render, alphas, gt_rgb, gt_rgb_is_u8, gt_depth, gt_depth_is_u16, depth_unit_scale, mask, mask_is_u8, bg,
                              rgb_weight, depth_lambda, ssim_lambda, grad_scale, stats_dev, loss_dev, v_render, v_alphas, bla, v_grid_rows, workspace,
                              workspace_bytes, (cudaStream_t)stream_);
}

extern "C" int qed_adam_arena(int64_t n, float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int G,
                              const int64_t* group_ends, const float* lr_by_group, const float* lr_alt_by_group,
                              const int32_t* group_period, const int32_t* group_split, double beta1, double beta2, double eps,
                              int step, qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n < 0 || G <= 0 || G > 16 || step < 1) return QED_ERR_BAD_ARG;
    if (n == 0) return QED_OK;
    if (!param || !grad || !exp_avg || !exp_avg_sq || !group_ends || !lr_by_group) return QED_ERR_BAD_ARG;
    // bias corrections in double, as torch.optim.Adam computes them on the host
    const float inv_bias1 = (float)(1.0 / (1.0 - pow(beta1, (double)step)));
    const float inv_bias2_sqrt = (float)(1.0 / sqrt(1.0 - pow(beta2, (double)step)));
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    const bool vec = (n % 4 == 0) && al16(param) && al16(grad) && al16(exp_avg) && al16(exp_avg_sq);
    if (vec) {
        const int64_t threads = (n / 4 + 1) / 2;  // two float4 per thread
        QED_CUDA_TRY(launch_pdl(adam_arena_kernel<true>, dim3((unsigned)((threads + 255) / 256)), dim3(256), 0, stream, n, param, grad, exp_avg, exp_avg_sq, G,
                                group_ends, lr_by_group, lr_alt_by_group, group_period, group_split, (float)beta1, (float)beta2, (float)eps,
                                inv_bias1, inv_bias2_sqrt));
    } else {
        QED_CUDA_TRY(launch_pdl(adam_arena_kernel<false>, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, stream, n, param, grad, exp_avg, exp_avg_sq, G,
                                group_ends, lr_by_group, lr_alt_by_group, group_period, group_split, (float)beta1, (float)beta2, (float)eps,
                                inv_bias1, inv_bias2_sqrt));
    }
    return QED_OK;
}

extern "C" int qed_strategy_update(int C, int N, const float* packed_grads, int use_absgrad, const int32_t* radii,
                                   int width, int height, int n_cameras, float* grad2d, float* count, float* radii_max,
                                   qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (C < 0 || N < 0 || width <= 0 || height <= 0) return QED_ERR_BAD_ARG;
    if (C == 0 || N == 0) return QED_OK;
    if (!packed_grads || !radii || !grad2d || !count) return QED_ERR_BAD_ARG;
    if (n_cameras <= 0) n_cameras = C;
    const float sx = (float)width / 2.0f * (float)n_cameras, sy = (float)height / 2.0f * (float)n_cameras;
    const float inv = 1.0f / (float)(width > height ? width : height);
    QED_CUDA_TRY(launch_pdl(strategy_update_kernel, dim3((N + 255) / 256), dim3(256), 0, stream, C, N, reinterpret_cast<const float4*>(packed_grads),
                            use_absgrad, radii, sx, sy, inv, grad2d, count, radii_max));
    return QED_OK;
}

// ------------------------------------------------------------------------------------------------
// densify / prune as one gather: 16 lanes per output Gaussian -- lanes 0..11 move the SH row (12 x float4 = 192 B,
// coalesced), lanes 12..15 the means / quats / log-scales / logit-opacity -- for the parameter arena and both
// Adam-moment arenas.  ~3 x 236 B read + written per Gaussian, nothing else.
// ------------------------------------------------------------------------------------------------
struct ArenaStarts {
    int64_t g[5];
};

__global__ void __launch_bounds__(256) arena_gather_kernel(int64_t n_new, const int32_t* __restrict__ src, const uint8_t* __restrict__ fresh,
                                                           const int32_t* __restrict__ child_row, const float* __restrict__ child_means,
                                                           const float* __restrict__ child_scales, const float* __restrict__ op,
                                                           const float* __restrict__ om, const float* __restrict__ ov, ArenaStarts os,
                                                           float* __restrict__ np, float* __restrict__ nm, float* __restrict__ nv, ArenaStarts ns) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t j = t >> 4;
    const int l = (int)(t & 15);
    if (j >= n_new) return;
    const int64_t s = src[j];
    const bool fr = fresh && fresh[j];
    const int cr = child_row ? child_row[j] : -1;
    if (l < 12) {
        const int64_t so = os.g[4] + s * 48 + l * 4, d = ns.g[4] + j * 48 + l * 4;
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4*>(np + d) = *reinterpret_cast<const float4*>(op + so);
        *reinterpret_cast<float4*>(nm + d) = fr ? z : *reinterpret_cast<const float4*>(om + so);
        *reinterpret_cast<float4*>(nv + d) = fr ? z : *reinterpret_cast<const float4*>(ov + so);
        return;
    }
    const int grp = l - 12;                        // 0 means, 1 quats, 2 log-scales, 3 logit-opacity
    const int dim = grp == 1 ? 4 : (grp == 3 ? 1 : 3);
    const int64_t so = os.g[grp] + s * dim, d = ns.g[grp] + j * dim;
    const float* over = (cr >= 0 && grp == 0) ? child_means + (int64_t)cr * 3 : ((cr >= 0 && grp == 2) ? child_scales + (int64_t)cr * 3 : nullptr);
    for (int k = 0; k < dim; ++k) {
        np[d + k] = over ? over[k] : op[so + k];
        nm[d + k] = fr ? 0.0f : om[so + k];
        nv[d + k] = fr ? 0.0f : ov[so + k];
    }
}

extern "C" int qed_arena_gather(int64_t n_new, const int32_t* src, const uint8_t* fresh, const int32_t* child_row,
                                const float* child_means, const float* child_scales, const float* old_param,
                                const float* old_exp_avg, const float* old_exp_avg_sq, const int64_t* old_group_starts,
                                float* new_param, float* new_exp_avg, float* new_exp_avg_sq, const int64_t* new_group_starts,
                                qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n_new < 0) return QED_ERR_BAD_ARG;
    if (n_new == 0) return QED_OK;
    if (!src || !old_param || !old_exp_avg || !old_exp_avg_sq || !old_group_starts || !new_param || !new_exp_avg || !new_exp_avg_sq ||
        !new_group_starts)
        return QED_ERR_BAD_ARG;
    if (child_row && (!child_means || !child_scales)) return QED_ERR_BAD_ARG;
    if (n_new > 0x7fffffffLL) return QED_ERR_UNSUPPORTED;
    ArenaStarts os, ns;
    for (int i = 0; i < 5; ++i) {
        os.g[i] = old_group_starts[i];
        ns.g[i] = new_group_starts[i];
    }
    auto mis = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) != 0; };
    if ((os.g[4] & 3) || (ns.g[4] & 3) || mis(old_param) || mis(old_exp_avg) || mis(old_exp_avg_sq) || mis(new_param) || mis(new_exp_avg) ||
        mis(new_exp_avg_sq))
        return QED_ERR_BAD_ARG;  // float4 access to the SH rows
    const int64_t threads = n_new * 16;
    arena_gather_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(n_new, src, fresh, child_row, child_means, child_scales, old_param,
                                                                             old_exp_avg, old_exp_avg_sq, os, new_param, new_exp_avg,
                                                                             new_exp_avg_sq, ns);
    QED_LAUNCH_CHECK();
    return QED_OK;
}

extern "C" int qed_abi_version(void) { return QED_ABI_VERSION; }

extern "C" const char* qed_error_string(int code) {
    switch (code) {
        case QED_OK: return "ok";
        case QED_ERR_BAD_ARG: return "qed: bad argument (null pointer, negative extent or inconsistent shape)";
        case QED_ERR_UNSUPPORTED: return "qed: unsupported configuration (tile_size != 16, D not in {1,3,4}, sh_degree > 3, or extent too large)";
        case QED_ERR_WORKSPACE: return "qed: workspace too small";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "qed: unknown error";
    }
}
