// Shared helpers for the sm_100a kernels of the splat hot path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "qed_splat.h"

#define QED_CUDA_TRY(expr)                       \
    do {                                         \
        cudaError_t _e = (expr);                 \
        if (_e != cudaSuccess) return (int)_e;   \
    } while (0)

#define QED_LAUNCH_CHECK()                        \
    do {                                          \
        cudaError_t _e = cudaPeekAtLastError();   \
        if (_e != cudaSuccess) return (int)_e;    \
    } while (0)

#include <cstdlib>
#include <utility>

namespace qed {

// ---- programmatic dependent launch (sm_90+): a step is a chain of ~23 mostly short kernels on one stream.  Every
// hot-path kernel starts with pdl_enter(): `griddepcontrol.launch_dependents` lets the NEXT kernel of the stream be
// scheduled as soon as every CTA of this one has started (its CTAs then fill the slots this kernel's tail leaves
// empty), `griddepcontrol.wait` holds this kernel until every kernel before it has completed and flushed -- nothing of a
// predecessor is read, and nothing it may still read is written, before that.  Launches go through launch_pdl(), which
// sets cudaLaunchAttributeProgrammaticStreamSerialization; QED_PDL=0 in the environment turns the attribute off (A/B).
__device__ __forceinline__ void pdl_enter() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

inline bool pdl_enabled() {
    static const bool on = [] {
        const char* e = std::getenv("QED_PDL");
        return !(e && e[0] == '0');
    }();
    return on;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...);
}

constexpr float kAlphaThreshold = 1.0f / 255.0f;
constexpr float kTransmittanceThreshold = 1e-4f;
constexpr float kMaxAlpha = 0.999f;
constexpr int kGeomFloats = 8;   // {mx,my,opacity,depth | conic a,b,c,0}
constexpr int kGradFloats = 12;  // {v_mx,v_my,|v_mx|,|v_my| | v_ca,v_cb,v_cc,v_op | v_colour[4]}

// Individually rounded IEEE ops: the projection mirrors the oracle's pinned op order exactly, so the
// compiler must never contract a*b+c into an FMA here (these intrinsics are never contracted).
__device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float dvd(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ float sqr(float a) { return __fsqrt_rn(a); }
// a*b + c*d, a*b - c*d with the oracle's rounding (two products, one sum)
__device__ __forceinline__ float mad2(float a, float b, float c, float d) { return add(mul(a, b), mul(c, d)); }
__device__ __forceinline__ float msb2(float a, float b, float c, float d) { return sub(mul(a, b), mul(c, d)); }
// (a*b + c*d) + e*f
__device__ __forceinline__ float mad3(float a, float b, float c, float d, float e, float f) {
    return add(add(mul(a, b), mul(c, d)), mul(e, f));
}

// Ground-truth image as the data side holds it: float32 in [0,1], or the uint8 cache of nerfstudio's
// FullImageDatamanager (qed_splatter/config.py:37 cache_images_type="uint8"), converted as splatfacto does
// (`image.float() / 255.0`) at the point of use instead of materialising a float copy per step.
struct GtImage {
    const void* p;
    int u8;
    __device__ __forceinline__ float at(int64_t i) const {
        // torch's CUDA `tensor / scalar` is `tensor * (1 / scalar)` in float: the same here, bit for bit
        return u8 ? __fmul_rn((float)reinterpret_cast<const uint8_t*>(p)[i], 1.0f / 255.0f) : reinterpret_cast<const float*>(p)[i];
    }
};

// Ground-truth depth as the data side holds it: float32 metres, or the raw uint16 sensor image (millimetres for the
// reference's datasets) with the unit scale of qed_splatter/dataparser.py:15 (depth_unit_scale_factor = 0.001, times the
// dataparser's scene scale) applied at the point of use -- nerfstudio's loader computes `image.astype(float64) * scale`,
// which is what `at()` returns, rounded to float32.  Keeps the depth cache at 2 B/pixel and removes a preprocessing pass.
struct GtDepth {
    const void* p;
    int u16;
    double scale;
    __device__ __forceinline__ float at(int64_t pix) const {
        return u16 ? (float)((double)reinterpret_cast<const uint16_t*>(p)[pix] * scale) : reinterpret_cast<const float*>(p)[pix];
    }
};

// Per-block partial sums of the held-out metrics pass (ssim.cu, SsimEval), summed per view by metrics.cu.
constexpr int kEvalPartials = 10;

// Optional per-pixel loss mask of the batch (`batch["mask"]`, qed_splatter/model.py:93-97; splatfacto multiplies the
// RGB images by it too): float32 or uint8 / bool [C,H,W]; NULL = all ones.
struct PixelMask {
    const void* p;
    int u8;
    __device__ __forceinline__ float at(int64_t pix) const {
        if (!p) return 1.0f;
        return u8 ? (float)reinterpret_cast<const uint8_t*>(p)[pix] : reinterpret_cast<const float*>(p)[pix];
    }
};

// ---- log2-domain alpha test shared by the compositor (raster.cu) and the exact tile lists (isect.cu) ----
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLog2_255 = 7.99435343685886f;

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Conservative test in the log2 domain: Q(d) = A dx^2 + B dx dy + C dy^2 (positive definite,
// = log2(e) * sigma), d = mean - pixel centre.  A pixel can only be touched if Q <= tau2 = lo + log2(255).
// Returns false only if the minimum of Q over the rectangle [x0,x1]x[y0,y1] exceeds tau2 by a margin.
__device__ __forceinline__ bool ellipse_hits_rect(float mx, float my, float A, float B, float C, float tau2, float x0, float y0,
                                                  float x1, float y1) {
    if (!(tau2 >= 0.0f)) return false;  // opacity < 1/255 can never pass the alpha test
    const float dxl = mx - x1, dxh = mx - x0;  // dx in [dxl, dxh]
    const float dyl = my - y1, dyh = my - y0;
    if (dxl <= 0.0f && dxh >= 0.0f && dyl <= 0.0f && dyh >= 0.0f) return true;  // centre inside
    // convex quadratic, centre outside: the minimum over the rectangle lies on an edge
    float best = 3.0e38f, mag = 0.0f;
    const float hC = 0.5f * rcp_approx(C), hA = 0.5f * rcp_approx(A);
#pragma unroll
    for (int e = 0; e < 2; ++e) {  // edges dx = const
        const float dx = e ? dxh : dxl;
        const float dy = fminf(fmaxf(-B * dx * hC, dyl), dyh);
        const float t0 = A * dx * dx, t1 = C * dy * dy, t2 = B * dx * dy;
        const float s = t0 + t1 + t2;
        if (s < best) {
            best = s;
            mag = t0 + t1 + fabsf(t2);
        }
    }
#pragma unroll
    for (int e = 0; e < 2; ++e) {  // edges dy = const
        const float dy = e ? dyh : dyl;
        const float dx = fminf(fmaxf(-B * dy * hA, dxl), dxh);
        const float t0 = A * dx * dx, t1 = C * dy * dy, t2 = B * dx * dy;
        const float s = t0 + t1 + t2;
        if (s < best) {
            best = s;
            mag = t0 + t1 + fabsf(t2);
        }
    }
    // margin: 1 % + absolute + rounding of the three terms (cancellation for thin, tilted ellipses)
    return !(best > tau2 * 1.01f + 0.03f + 2e-5f * mag);
}

// ---- EXACT tile lists: which tiles of a Gaussian's 3-sigma bounding box can be touched at all -------------------------
// A Gaussian changes a pixel only if alpha >= 1/255, i.e. the pixel centre lies in the ellipse Q(mean - p) <= tau2,
// Q = A dx^2 + B dx dy + C dy^2 (the compositor's log2 domain), tau2 = log2(255 opacity).  For one TILE ROW (a horizontal
// strip ya <= y <= yb of pixel centres) the part of the ellipse inside the strip is convex, so the tiles of that row that
// can be touched form ONE interval of tile columns [c0, c1):
//   fixed dy: A dx^2 + B dy dx + C dy^2 - t <= 0  ->  dx in (-B dy -+ sqrt(disc)) / 2A,  disc = 4 A t - det dy^2,  det = 4AC - B^2
//   the right end dx_hi(dy) is concave with its maximum dxmax = sqrt(4 C t / det) at dy = -B dxmax / 2C, the left end mirrors it.
// exact_ctx() is evaluated once per Gaussian, exact_row_span() once per (Gaussian, tile row).  The projection kernel SUMS
// the spans (the exact tile count that is scanned into the list offsets) and the emit kernel ENUMERATES them, so both must
// produce identical integers: every float operation below is an explicitly rounded intrinsic or a hardware approximation
// instruction (no contraction, no compiler-dependent reassociation).  Conservative: tau2 is inflated as in
// ellipse_hits_rect and the interval is widened by 0.1 px + 0.5 % of the ellipse's half-width (cancellation in det for
// thin, tilted ellipses); the compositor keeps its own per-warp test, so a tile too many costs time, never a pixel.
__device__ __forceinline__ float rsqrt_approx(float x) {
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

struct ExactCtx {
    float mx, my, negB, det, fourAt, dymax, dys, r2A, slack;
    bool valid;  // false: opacity < 1/255, the Gaussian can never pass the alpha test
};

__device__ __forceinline__ ExactCtx exact_ctx(float mx, float my, float opacity, float ca, float cb, float cc) {
    ExactCtx e;
    const float A = mul(0.5f * kLog2e, ca), B = mul(kLog2e, cb), C = mul(0.5f * kLog2e, cc);
    const float tau2 = add(lg2_approx(opacity), kLog2_255);
    const float t = add(mul(tau2, 1.01f), 0.03f);
    e.valid = tau2 >= 0.0f;
    e.mx = mx;
    e.my = my;
    e.negB = -B;
    e.det = fmaxf(sub(mul(mul(4.0f, A), C), mul(B, B)), 1e-30f);
    const float rdet = rcp_approx(e.det);
    e.fourAt = mul(mul(4.0f, A), t);
    const float ey = mul(e.fourAt, rdet), ex = mul(mul(mul(4.0f, C), t), rdet);  // squared half-extents in y / x
    e.dymax = add(mul(mul(ey, rsqrt_approx(fmaxf(ey, 1e-30f))), 1.0001f), 1e-3f);  // sqrt(e) = e * rsqrt(e)
    const float dxmax = mul(ex, rsqrt_approx(fmaxf(ex, 1e-30f)));
    e.dys = mul(mul(mul(-0.5f, B), dxmax), rcp_approx(C));  // dy of the right extreme point (the left one sits at -dys)
    e.r2A = mul(0.5f, rcp_approx(A));
    e.slack = add(0.1f, mul(0.005f, dxmax));
    return e;
}

// tile columns [c0, c1) (inside the bounding box columns [bx0, bx1)) of tile row `ty` that the ellipse can touch; 16-pixel tiles
__device__ __forceinline__ void exact_row_span(const ExactCtx& e, int ty, int height, int bx0, int bx1, int& c0, int& c1) {
    const float ya = (float)(ty * 16) + 0.5f, yb = (float)min(ty * 16 + 15, height - 1) + 0.5f;
    const float dl = fmaxf(sub(e.my, yb), -e.dymax), dh = fminf(sub(e.my, ya), e.dymax);  // dy = my - y over the strip, cut to the ellipse
    const float dy_hi = fminf(fmaxf(e.dys, dl), dh), dy_lo = fminf(fmaxf(-e.dys, dl), dh);
    const float disc_hi = fmaxf(sub(e.fourAt, mul(e.det, mul(dy_hi, dy_hi))), 0.0f);
    const float disc_lo = fmaxf(sub(e.fourAt, mul(e.det, mul(dy_lo, dy_lo))), 0.0f);
    const float s_hi = mul(disc_hi, rsqrt_approx(fmaxf(disc_hi, 1e-30f))), s_lo = mul(disc_lo, rsqrt_approx(fmaxf(disc_lo, 1e-30f)));
    const float dx_hi = mul(add(mul(e.negB, dy_hi), s_hi), e.r2A), dx_lo = mul(sub(mul(e.negB, dy_lo), s_lo), e.r2A);
    const float xlo = sub(sub(e.mx, dx_hi), e.slack), xhi = add(sub(e.mx, dx_lo), e.slack);  // x = mx - dx
    // tile column tx has pixel centres [16 tx + 0.5, 16 tx + 15.5] (the clipped last column is treated as full: conservative)
    const float f0 = fminf(fmaxf(ceilf(mul(sub(xlo, 15.5f), 0.0625f)), (float)bx0), (float)bx1);
    const float f1 = fminf(fmaxf(add(floorf(mul(sub(xhi, 0.5f), 0.0625f)), 1.0f), (float)bx0), (float)bx1);
    const bool hit = e.valid && (dl <= dh) && (f1 > f0);
    c0 = (int)f0;
    c1 = hit ? (int)f1 : c0;
}

// ---- packed float pairs (sm_100 FFMA2 / FMUL2 / FADD2: one issue slot, two IEEE fp32 results) -------------
// ptxas folds bc2(s) into a scalar-broadcast operand (`R.F32`), neg2/abs2 into operand modifiers and pk2 of
// two freshly produced scalars into adjacent registers, so these helpers cost no extra instructions.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ f32x2 bc2(float s) { return pk2(s, s); }
__device__ __forceinline__ float lo2(f32x2 v) {
    float a, b;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
    return a;
}
__device__ __forceinline__ float hi2(f32x2 v) {
    float a, b;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
    return b;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 neg2(f32x2 v) { return pk2(-lo2(v), -hi2(v)); }
__device__ __forceinline__ f32x2 abs2(f32x2 v) { return pk2(fabsf(lo2(v)), fabsf(hi2(v))); }

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

__device__ __forceinline__ float4 ldg_nc_f4(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void red_add_v2(float* addr, float a, float b) {
    asm volatile("red.global.add.v2.f32 [%0], {%1,%2};" ::"l"(addr), "f"(a), "f"(b) : "memory");
}

struct TileBox {
    int x0, y0, x1, y1;  // [x0,x1) x [y0,y1)
};

// gsplat isect_tiles: tile_min = floor(mean/ts - r/ts), tile_max = ceil(mean/ts + r/ts), clamped to the grid.
__device__ __forceinline__ TileBox tile_box(float mx, float my, int radius, float tile_size, int tile_width,
                                            int tile_height) {
    float tr = dvd((float)radius, tile_size);
    float tx = dvd(mx, tile_size);
    float ty = dvd(my, tile_size);
    // clamp in float first so the int conversion cannot overflow
    float fx0 = fminf(fmaxf(floorf(sub(tx, tr)), 0.0f), (float)tile_width);
    float fy0 = fminf(fmaxf(floorf(sub(ty, tr)), 0.0f), (float)tile_height);
    float fx1 = fminf(fmaxf(ceilf(add(tx, tr)), 0.0f), (float)tile_width);
    float fy1 = fminf(fmaxf(ceilf(add(ty, tr)), 0.0f), (float)tile_height);
    TileBox b;
    b.x0 = (int)fx0;
    b.y0 = (int)fy0;
    b.x1 = (int)fx1;
    b.y1 = (int)fy1;
    return b;
}

}  // namespace qed
