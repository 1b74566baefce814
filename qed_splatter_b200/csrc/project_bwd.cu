// (a) backward of the fused projection + SH colour stage.
//
// Replaces gsplat's fully_fused_projection_bwd + compute_sh_bwd + the glue VJPs (clamp_min(c+0.5),
// depth-channel concat, opacity*compensation) behind qed_splatter/model.py:267-288's autograd.
// Semantics: SURVEY.md Appendix A.7, hand-derived VJP of oracle/torch_impl.py::fully_fused_projection /
// spherical_harmonics; parity is against torch autograd of that oracle (tests/test_project.py).
//
// Mapping: one thread per Gaussian, cameras looped inside (so the per-camera sum needs no atomics and is
// deterministic).  SH coefficients are staged warp-cooperatively into shared memory (cp.async, 16 B,
// rows padded to an odd float4 count) and the 192 B/Gaussian coefficient gradient is built in a second
// padded buffer and streamed out with coalesced 16-byte stores.
// HBM-bound: ~48 B packed grads + 236 B inputs read and 236 B gradients written per Gaussian.
#include "common.cuh"

namespace qed {

constexpr int kProjBwdThreads = 128;
constexpr int kCamFloatsB = 32;

struct CamB {
    float W[9];
    float t[3];
    float fx, fy, cx, cy;
    float lim_xp, lim_xn, lim_yp, lim_yn;
    float campos[3];
    float pad[9];
};

struct ProjBwdParams {
    int C, N, K, sh_degree, colors_per_camera, width, height;
    float eps2d;
    int calc_comp, n_color, append_depth, activations;
    const float *means, *quats, *scales, *opacities, *colors_in, *viewmats, *Ks;
    const int32_t* radii;
    const float *conics, *comps;
    const float *v_means2d, *v_depths, *v_conics, *v_colors, *v_opac_cn, *packed;
    float *v_means, *v_quats, *v_scales, *v_opacities, *v_colors_in;
    // view-colour exchange (multi-GPU, see qed_project_bwd_exchange): instead of the 192-B SH coefficient gradient, the
    // gated colour gradient of every VISIBLE (view, Gaussian) is stored as {v_r, v_g, v_b, tag} into slot
    // (xch_slot0 + c) * N + n of the exchange buffer of every rank
    float4* xch_mc;                // NVSwitch multicast address of the exchange buffer, or NULL
    float4* xch_peer[16];          // else: its unicast address on every rank
    int xch_world, xch_slot0, xch_total_slots;
    float xch_tag;
    // camera pose gradient (POSE, see qed_project_bwd_pose / qed_project_bwd_exchange_pose): per-warp partial sums of the 15 per-view values
    // {v_W (9, row-major), v_t (3), sum of the SH direction gradient (3), 0}, 4 float4 at (c * warps + warp) * 4
    float4* pose_ws;
};

constexpr int kPoseVals = 15;

// Sums the 15 per-view pose values of the warp's 32 Gaussians (butterfly: a fixed order, every lane ends with the same
// bits) and stores them as the warp's partial of view c.  The values live in shared memory, [kPoseVals][kProjBwdThreads],
// each thread touching only its own column (registers would spill in the degree-3 kernels); the column is cleared for
// the next view.  Every lane of the warp must call it at the same point.
__device__ __forceinline__ void pose_flush(const ProjBwdParams& p, int c, float* pose_s) {
    float* dst = reinterpret_cast<float*>(p.pose_ws + ((int64_t)c * gridDim.x * (kProjBwdThreads / 32) + blockIdx.x * (kProjBwdThreads / 32) +
                                                       (threadIdx.x >> 5)) * 4);
#pragma unroll
    for (int k = 0; k < kPoseVals; ++k) {
        float v = pose_s[k * kProjBwdThreads + threadIdx.x];
        pose_s[k * kProjBwdThreads + threadIdx.x] = 0.0f;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if ((threadIdx.x & 31) == 0) dst[k] = v;
    }
    if ((threadIdx.x & 31) == 0) dst[kPoseVals] = 0.0f;
}

__device__ __forceinline__ void xch_store(const ProjBwdParams& p, int64_t i, float4 v) {
    if (p.xch_mc) {
        asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p.xch_mc + i), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
    } else {
        for (int r = 0; r < p.xch_world; ++r) p.xch_peer[r][i] = v;
    }
}

__device__ void load_camera_b(const float* __restrict__ V, const float* __restrict__ Kc, int width, int height, CamB& cam) {
    float a[3][3], t[3];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) {
            a[i][j] = V[i * 4 + j];
            cam.W[i * 3 + j] = a[i][j];
        }
        t[i] = V[i * 4 + 3];
        cam.t[i] = t[i];
    }
    float fx = Kc[0], fy = Kc[4], cx = Kc[2], cy = Kc[5];
    cam.fx = fx;
    cam.fy = fy;
    cam.cx = cx;
    cam.cy = cy;
    float tanx = 0.5f * (float)width / fx, tany = 0.5f * (float)height / fy;
    cam.lim_xp = ((float)width - cx) / fx + 0.3f * tanx;
    cam.lim_xn = cx / fx + 0.3f * tanx;
    cam.lim_yp = ((float)height - cy) / fy + 0.3f * tany;
    cam.lim_yn = cy / fy + 0.3f * tany;
    float c00 = a[1][1] * a[2][2] - a[1][2] * a[2][1], c01 = a[0][2] * a[2][1] - a[0][1] * a[2][2], c02 = a[0][1] * a[1][2] - a[0][2] * a[1][1];
    float c10 = a[1][2] * a[2][0] - a[1][0] * a[2][2], c11 = a[0][0] * a[2][2] - a[0][2] * a[2][0], c12 = a[0][2] * a[1][0] - a[0][0] * a[1][2];
    float c20 = a[1][0] * a[2][1] - a[1][1] * a[2][0], c21 = a[0][1] * a[2][0] - a[0][0] * a[2][1], c22 = a[0][0] * a[1][1] - a[0][1] * a[1][0];
    float det = a[0][0] * c00 + a[0][1] * c10 + a[0][2] * c20;
    cam.campos[0] = -(c00 * t[0] + c01 * t[1] + c02 * t[2]) / det;
    cam.campos[1] = -(c10 * t[0] + c11 * t[1] + c12 * t[2]) / det;
    cam.campos[2] = -(c20 * t[0] + c21 * t[1] + c22 * t[2]) / det;
}

template <int DEG>
struct ShShapeB {
    static constexpr int kBases = (DEG + 1) * (DEG + 1);
    static constexpr int kFloats = 3 * kBases;
    static constexpr int kVec = (kFloats + 3) / 4;
    static constexpr int kStrideVec = (kVec % 2) ? kVec : kVec + 1;
};

// bases and the VJP d(sum_k vb[k] b_k)/d(x,y,z) for a unit direction
template <int DEG>
__device__ __forceinline__ void sh_bases_b(float x, float y, float z, float* b) {
    b[0] = 0.2820947917738781f;
    if (DEG >= 1) {
        b[1] = -0.48860251190292f * y;
        b[2] = 0.48860251190292f * z;
        b[3] = -0.48860251190292f * x;
    }
    if (DEG >= 2) {
        float z2 = z * z, fTmp0B = -1.092548430592079f * z, fC1 = x * x - y * y, fS1 = 2.0f * x * y;
        b[4] = 0.5462742152960395f * fS1;
        b[5] = fTmp0B * y;
        b[6] = 0.9461746957575601f * z2 - 0.3153915652525201f;
        b[7] = fTmp0B * x;
        b[8] = 0.5462742152960395f * fC1;
        if (DEG >= 3) {
            float fTmp0C = -2.285228997322329f * z2 + 0.4570457994644658f, fTmp1B = 1.445305721320277f * z;
            float fC2 = x * fC1 - y * fS1, fS2 = x * fS1 + y * fC1;
            b[9] = -0.5900435899266435f * fS2;
            b[10] = fTmp1B * fS1;
            b[11] = fTmp0C * y;
            b[12] = z * (1.865881662950577f * z2 - 1.119528997770346f);
            b[13] = fTmp0C * x;
            b[14] = fTmp1B * fC1;
            b[15] = -0.5900435899266435f * fC2;
        }
    }
}

template <int DEG>
__device__ __forceinline__ void sh_bases_vjp(float x, float y, float z, const float* vb, float& vx, float& vy, float& vz) {
    vx = vy = vz = 0.0f;
    if (DEG >= 1) {
        const float C1 = 0.48860251190292f;
        vx += -C1 * vb[3];
        vy += -C1 * vb[1];
        vz += C1 * vb[2];
    }
    if (DEG >= 2) {
        const float A = -1.092548430592079f, P = 0.5462742152960395f, Q = 0.9461746957575601f;
        vx += 2.0f * P * y * vb[4] + A * z * vb[7] + 2.0f * P * x * vb[8];
        vy += 2.0f * P * x * vb[4] + A * z * vb[5] - 2.0f * P * y * vb[8];
        vz += A * y * vb[5] + 2.0f * Q * z * vb[6] + A * x * vb[7];
    }
    if (DEG >= 3) {
        const float E = -2.285228997322329f, F = 0.4570457994644658f, G = 1.445305721320277f;
        const float H = -0.5900435899266435f, U = 1.865881662950577f, V = 1.119528997770346f;
        float z2 = z * z, fC1 = x * x - y * y, fS1 = 2.0f * x * y, fTmp0C = E * z2 + F;
        vx += 3.0f * H * fS1 * vb[9] + 2.0f * G * y * z * vb[10] + fTmp0C * vb[13] + 2.0f * G * z * x * vb[14] + 3.0f * H * fC1 * vb[15];
        vy += 3.0f * H * fC1 * vb[9] + 2.0f * G * x * z * vb[10] + fTmp0C * vb[11] - 2.0f * G * z * y * vb[14] - 3.0f * H * fS1 * vb[15];
        vz += G * fS1 * vb[10] + 2.0f * E * z * y * vb[11] + (3.0f * U * z2 - V) * vb[12] + 2.0f * E * z * x * vb[13] + G * fC1 * vb[14];
    }
}

__device__ __forceinline__ void quat_to_rotmat(float qw, float qx, float qy, float qz, float (&R)[9]) {
    R[0] = 1.0f - 2.0f * (qy * qy + qz * qz);
    R[1] = 2.0f * (qx * qy - qw * qz);
    R[2] = 2.0f * (qx * qz + qw * qy);
    R[3] = 2.0f * (qx * qy + qw * qz);
    R[4] = 1.0f - 2.0f * (qx * qx + qz * qz);
    R[5] = 2.0f * (qy * qz - qw * qx);
    R[6] = 2.0f * (qx * qz - qw * qy);
    R[7] = 2.0f * (qy * qz + qw * qx);
    R[8] = 1.0f - 2.0f * (qx * qx + qy * qy);
}

// DEG=-1: colours pass through.  VEC: coefficient rows 16-byte aligned and K*3 % 4 == 0.
// XCH (multi-GPU view-colour exchange, VEC only): no coefficient gradient is built or written (half the shared memory, 192 B
// per Gaussian less HBM traffic); the gated colour gradient goes to every rank's exchange buffer instead.
// ONE (a single view, VEC only -- the reference's case, model.py:211): the coefficient gradient b (x) vpre needs no sum over
// views, so it overwrites the staged coefficient row in place: half the shared memory, and with it 5 resident blocks per SM
// instead of 4 (the kernel is latency-bound: 35 % issue-active at 16 warps per SM).  ONE = resident blocks asked of ptxas (5: 96
// registers, 6: 80 registers).
// POSE: also the gradient with respect to each view's world-to-camera matrix [W | t].  For every visible
// (view, Gaussian) the values below are already in registers: the camera-space mean gradient v_p, the camera-space
// covariance gradient vSc with A = W Sigma, and the SH direction gradient v_d.  v_W += v_p mu^T + 2 vSc A, v_t += v_p,
// and sum v_d is kept for the camera-position term, which pose_finish_kernel applies once per view.  Per-warp partials
// (pose_flush) at the end for ONE, after every view otherwise: the view loop then runs in every lane of the warp.  With XCH
// the direction gradient comes from the same vb the exchange branch builds, so the pose values are the same.
template <int DEG, bool VEC, bool XCH = false, int ONE = 0, bool POSE = false>
__global__ void __launch_bounds__(kProjBwdThreads, ONE ? ONE : 4) project_bwd_kernel(const ProjBwdParams p) {
    extern __shared__ float4 smem4[];
    pdl_enter();
    const int nC = ONE ? 1 : p.C;  // ONE: the view loops collapse at compile time
    CamB* cams = reinterpret_cast<CamB*>(smem4);
    constexpr int DG = DEG < 0 ? 0 : DEG;
    using Sh = ShShapeB<DG>;
    float* pose_s = reinterpret_cast<float*>(smem4 + nC * (kCamFloatsB / 4));  // POSE: [kPoseVals][kProjBwdThreads]
    float4* coefbuf = smem4 + nC * (kCamFloatsB / 4) + (POSE ? kPoseVals * kProjBwdThreads / 4 : 0);
    float4* vcoefbuf = ONE ? coefbuf : coefbuf + kProjBwdThreads * Sh::kStrideVec;

    for (int c = threadIdx.x; c < nC; c += kProjBwdThreads) load_camera_b(p.viewmats + c * 16, p.Ks + c * 9, p.width, p.height, cams[c]);
    __syncthreads();

    const int n = blockIdx.x * kProjBwdThreads + threadIdx.x;
    const bool in_range = n < p.N;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int D = p.n_color + p.append_depth;
    const bool use_sh = DEG >= 0 && p.n_color > 0;

    // Every global load of this Gaussian is ISSUED before the first one is used (the kernel runs 16 warps per SM, so a
    // chain of dependent round trips -- inputs, radii, SH rows, packed gradients, conics -- is what bounds it): radii first
    // (they gate the SH staging), then the raw parameters, then the SH rows (cp.async) and the first view's upstream
    // gradients; the arithmetic on the parameters starts while those are in flight.
    float m0 = 0, m1 = 0, m2 = 0, s0 = 0, s1 = 0, s2 = 0, opac = 0, qn = 1;
    float qw = 1, qx = 0, qy = 0, qz = 0;
    float S00 = 0, S01 = 0, S02 = 0, S11 = 0, S12 = 0, S22 = 0;
    float4 q = make_float4(1.0f, 0.0f, 0.0f, 0.0f);
    bool anyvis = false;
    int rad0 = 0;
    if (in_range) {
        rad0 = p.radii[n];
        anyvis = rad0 > 0;
        for (int c = 1; c < nC; ++c) anyvis |= p.radii[(int64_t)c * p.N + n] > 0;
        m0 = p.means[n * 3 + 0];
        m1 = p.means[n * 3 + 1];
        m2 = p.means[n * 3 + 2];
        const float* qp = p.quats + (int64_t)n * 4;  // scalar loads: callers' views are only 4-byte aligned
        q = make_float4(qp[0], qp[1], qp[2], qp[3]);
        s0 = p.scales[n * 3 + 0];
        s1 = p.scales[n * 3 + 1];
        s2 = p.scales[n * 3 + 2];
        opac = p.opacities ? p.opacities[n] : 0.0f;
    }

    // ---- stage SH coefficients (visible rows) and clear the coefficient-gradient rows ----
    float4* my_coef = coefbuf + (warp * 32 + lane) * Sh::kStrideVec;
    float4* my_vcoef = vcoefbuf + (warp * 32 + lane) * Sh::kStrideVec;
    const int row_floats = p.K * 3;
    if (use_sh && VEC) {
        const uint32_t warp_vis = __ballot_sync(0xffffffffu, anyvis);
        const int64_t row0 = (int64_t)blockIdx.x * kProjBwdThreads + warp * 32;
        const float4* src = reinterpret_cast<const float4*>(p.colors_in) + row0 * (row_floats / 4);
        float4* wbuf = coefbuf + warp * 32 * Sh::kStrideVec;
        if (Sh::kVec == 12 && row_floats == 48) {
            // degree 3, K = 16: 4 lanes per row, 8 rows per step -- row / column are bit operations of the lane plus
            // compile-time constants (the generic loop below spends ~30 instructions per float4 on q / kVec and 64-bit
            // address arithmetic: 16 % of the kernel's instructions)
            const int r0 = lane >> 2, j0 = lane & 3;
            const float4* s0 = src + r0 * 12 + j0;
            float4* d0 = wbuf + r0 * Sh::kStrideVec + j0;
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
                if ((warp_vis >> (r0 + 8 * rr)) & 1u) {
#pragma unroll
                    for (int jj = 0; jj < 3; ++jj) cp_async16(d0 + rr * 8 * Sh::kStrideVec + 4 * jj, s0 + rr * 8 * 12 + 4 * jj);
                }
            }
        } else {
            for (int v = lane; v < 32 * Sh::kVec; v += 32) {
                int r = v / Sh::kVec, j = v - r * Sh::kVec;
                if ((warp_vis >> r) & 1u) cp_async16(wbuf + r * Sh::kStrideVec + j, src + (int64_t)r * (row_floats / 4) + j);
            }
        }
        cp_async_commit();
    }
    // upstream gradients + conic of the first view (the later views' are fetched one view ahead inside the loop)
    float4 pf0 = make_float4(0, 0, 0, 0), pf1 = pf0, pf2 = pf0;
    float pfa = 0, pfb = 0, pfc = 0;
    if (rad0 > 0) {
        if (p.packed) {
            const float4* r = reinterpret_cast<const float4*>(p.packed) + (int64_t)n * 3;
            pf0 = r[0];
            pf1 = r[1];
            pf2 = r[2];
        }
        pfa = p.conics[(int64_t)n * 3 + 0];
        pfb = p.conics[(int64_t)n * 3 + 1];
        pfc = p.conics[(int64_t)n * 3 + 2];
    }
    if (use_sh && !XCH && (!ONE || !anyvis)) {  // ONE: the rows of visible Gaussians are being filled by cp.async; nobody touches the others
#pragma unroll
        for (int j = 0; j < Sh::kVec; ++j) my_vcoef[j] = make_float4(0, 0, 0, 0);
    }
    if (in_range) {
        if (p.activations & QED_ACT_LOG_SCALES) {
            s0 = expf(s0);
            s1 = expf(s1);
            s2 = expf(s2);
        }
        if ((p.activations & QED_ACT_LOGIT_OPACITIES) && p.opacities) opac = 1.0f / (1.0f + expf(-opac));
        qn = fmaxf(sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w), 1e-12f);
        const float rqn = 1.0f / qn;  // one division, then products (IEEE `/` is a ~12-instruction sequence with a slow path)
        qw = q.x * rqn;
        qx = q.y * rqn;
        qy = q.z * rqn;
        qz = q.w * rqn;
        float R[9], M[9];  // R(q), M = R diag(s): rebuilt in the epilogue instead of living in 18 registers across the view loop
        quat_to_rotmat(qw, qx, qy, qz, R);
        for (int i = 0; i < 3; ++i) {
            M[i * 3 + 0] = R[i * 3 + 0] * s0;
            M[i * 3 + 1] = R[i * 3 + 1] * s1;
            M[i * 3 + 2] = R[i * 3 + 2] * s2;
        }
        S00 = M[0] * M[0] + M[1] * M[1] + M[2] * M[2];
        S01 = M[0] * M[3] + M[1] * M[4] + M[2] * M[5];
        S02 = M[0] * M[6] + M[1] * M[7] + M[2] * M[8];
        S11 = M[3] * M[3] + M[4] * M[4] + M[5] * M[5];
        S12 = M[3] * M[6] + M[4] * M[7] + M[5] * M[8];
        S22 = M[6] * M[6] + M[7] * M[7] + M[8] * M[8];
    }
    if (use_sh && VEC) {
        cp_async_wait<0>();
        __syncwarp();
    }

    float vS00 = 0, vS01 = 0, vS02 = 0, vS11 = 0, vS12 = 0, vS22 = 0;  // full symmetric matrix gradient (off-diag = one side)
    float vm0 = 0, vm1 = 0, vm2 = 0, vopac = 0;
    constexpr bool kWarpViews = POSE && !ONE;  // every lane runs the view loop (a warp reduction per view)
    if (POSE) {
#pragma unroll
        for (int k = 0; k < kPoseVals; ++k) pose_s[k * kProjBwdThreads + threadIdx.x] = 0.0f;
    }

    if (kWarpViews || (in_range && anyvis)) {
        int rad_c = rad0;
        for (int c = 0; c < nC; ++c) {
            if (kWarpViews && c > 0) pose_flush(p, c - 1, pose_s);
            const int64_t idx = (int64_t)c * p.N + n;
            const bool vis = rad_c > 0;
            const float4 r0 = pf0, r1 = pf1, r2 = pf2;
            const float ca = pfa, cb = pfb, cc = pfc;  // conic of the blurred covariance (stored by the forward)
            if (c + 1 < nC && (!kWarpViews || in_range)) {  // next view: radius, upstream gradients, conic
                const int64_t nx = idx + p.N;
                rad_c = p.radii[nx];
                if (rad_c > 0) {
                    if (p.packed) {
                        const float4* r = reinterpret_cast<const float4*>(p.packed) + nx * 3;
                        pf0 = r[0];
                        pf1 = r[1];
                        pf2 = r[2];
                    }
                    pfa = p.conics[nx * 3 + 0];
                    pfb = p.conics[nx * 3 + 1];
                    pfc = p.conics[nx * 3 + 2];
                }
            }
            if (!vis) continue;
            const CamB& cam = cams[c];
            const float* W = cam.W;
            // ---- incoming gradients ----
            float g_mx = 0, g_my = 0, g_d = 0, g_ca = 0, g_cb = 0, g_cc = 0, g_o = 0, g_col[4] = {0, 0, 0, 0};
            if (p.packed) {
                g_mx = r0.x;
                g_my = r0.y;
                g_ca = r1.x;
                g_cb = r1.y;
                g_cc = r1.z;
                g_o = r1.w;
                g_col[0] = r2.x;
                g_col[1] = r2.y;
                g_col[2] = r2.z;
                g_col[3] = r2.w;
            }
            if (p.v_means2d) {
                g_mx += p.v_means2d[idx * 2 + 0];
                g_my += p.v_means2d[idx * 2 + 1];
            }
            if (p.v_depths) g_d += p.v_depths[idx];
            if (p.v_conics) {
                g_ca += p.v_conics[idx * 3 + 0];
                g_cb += p.v_conics[idx * 3 + 1];
                g_cc += p.v_conics[idx * 3 + 2];
            }
            if (p.v_opac_cn) g_o += p.v_opac_cn[idx];
            if (p.v_colors) {
#pragma unroll
                for (int ch = 0; ch < 4; ++ch)
                    if (ch < D) g_col[ch] += p.v_colors[idx * D + ch];
            }
            if (p.append_depth) g_d += p.n_color == 3 ? g_col[3] : (p.n_color == 1 ? g_col[1] : g_col[0]);  // no dynamic index: registers

            // ---- recompute forward intermediates ----
            float x = W[0] * m0 + W[1] * m1 + W[2] * m2 + cam.t[0];
            float y = W[3] * m0 + W[4] * m1 + W[5] * m2 + cam.t[1];
            float z = W[6] * m0 + W[7] * m1 + W[8] * m2 + cam.t[2];
            float A[9];
            for (int i = 0; i < 3; ++i) {
                A[i * 3 + 0] = W[i * 3] * S00 + W[i * 3 + 1] * S01 + W[i * 3 + 2] * S02;
                A[i * 3 + 1] = W[i * 3] * S01 + W[i * 3 + 1] * S11 + W[i * 3 + 2] * S12;
                A[i * 3 + 2] = W[i * 3] * S02 + W[i * 3 + 1] * S12 + W[i * 3 + 2] * S22;
            }
            float Sc00 = A[0] * W[0] + A[1] * W[1] + A[2] * W[2];
            float Sc01 = A[0] * W[3] + A[1] * W[4] + A[2] * W[5];
            float Sc02 = A[0] * W[6] + A[1] * W[7] + A[2] * W[8];
            float Sc11 = A[3] * W[3] + A[4] * W[4] + A[5] * W[5];
            float Sc12 = A[3] * W[6] + A[4] * W[7] + A[5] * W[8];
            float Sc22 = A[6] * W[6] + A[7] * W[7] + A[8] * W[8];
            float rz = 1.0f / z, rz2 = rz * rz;
            float xz = x * rz, yz = y * rz;
            bool x_in = (xz <= cam.lim_xp) && (xz >= -cam.lim_xn);
            bool y_in = (yz <= cam.lim_yp) && (yz >= -cam.lim_yn);
            float tx = z * fmaxf(fminf(xz, cam.lim_xp), -cam.lim_xn);
            float ty = z * fmaxf(fminf(yz, cam.lim_yp), -cam.lim_yn);
            float J00 = cam.fx * rz, J02 = -cam.fx * tx * rz2, J11 = cam.fy * rz, J12 = -cam.fy * ty * rz2;

            // ---- conic -> blurred 2x2 covariance: G = -X V X, V = [[va, vb/2],[vb/2, vc]] ----
            float hv = 0.5f * g_cb;
            float XV00 = ca * g_ca + cb * hv, XV01 = ca * hv + cb * g_cc;
            float XV10 = cb * g_ca + cc * hv, XV11 = cb * hv + cc * g_cc;
            float G00 = -(XV00 * ca + XV01 * cb);
            float G01 = -(XV00 * cb + XV01 * cc);
            float G11 = -(XV10 * cb + XV11 * cc);
            // ---- opacity / compensation ----
            if (p.calc_comp) {
                float comp = p.comps[idx];
                vopac += g_o * comp;
                float v_comp = g_o * opac;
                float v_q = v_comp * 0.5f / (comp + 1e-6f);
                float omq = 1.0f - comp * comp;
                float detX = ca * cc - cb * cb;
                G00 += v_q * (omq * ca - p.eps2d * detX);
                G01 += v_q * (omq * cb);
                G11 += v_q * (omq * cc - p.eps2d * detX);
            } else {
                vopac += g_o;
            }
            // ---- cov2d = J Sc J^T ----
            // GJ (2x3) = G J ; vSc = J^T G J ; vJ = 2 G J Sc
            float GJ00 = G00 * J00, GJ01 = G01 * J11, GJ02 = G00 * J02 + G01 * J12;
            float GJ10 = G01 * J00, GJ11 = G11 * J11, GJ12 = G01 * J02 + G11 * J12;
            float vSc00 = J00 * GJ00;
            float vSc01 = J00 * GJ01;
            float vSc02 = J00 * GJ02;
            float vSc11 = J11 * GJ11;
            float vSc12 = J11 * GJ12;
            float vSc22 = J02 * GJ02 + J12 * GJ12;
            // symmetric counterparts: vSc10 = J11*GJ10 = vSc01 (G symmetric), etc.
            float vJ00 = 2.0f * (GJ00 * Sc00 + GJ01 * Sc01 + GJ02 * Sc02);
            float vJ02 = 2.0f * (GJ00 * Sc02 + GJ01 * Sc12 + GJ02 * Sc22);
            float vJ11 = 2.0f * (GJ10 * Sc01 + GJ11 * Sc11 + GJ12 * Sc12);
            float vJ12 = 2.0f * (GJ10 * Sc02 + GJ11 * Sc12 + GJ12 * Sc22);
            // ---- camera-space mean ----
            float vx = cam.fx * rz * g_mx;
            float vy = cam.fy * rz * g_my;
            float vz = -(cam.fx * x * g_mx + cam.fy * y * g_my) * rz2 + g_d;
            float rz3 = rz2 * rz;
            vz += -cam.fx * rz2 * vJ00 - cam.fy * rz2 * vJ11;
            if (x_in) {
                vx += -cam.fx * rz2 * vJ02;
                vz += 2.0f * cam.fx * tx * rz3 * vJ02;
            } else {
                vz += cam.fx * tx * rz3 * vJ02;
            }
            if (y_in) {
                vy += -cam.fy * rz2 * vJ12;
                vz += 2.0f * cam.fy * ty * rz3 * vJ12;
            } else {
                vz += cam.fy * ty * rz3 * vJ12;
            }
            if (POSE) {  // p = W mu + t and Sc = W Sigma W^T (vSc symmetric): v_W = v_p mu^T + 2 vSc A, v_t = v_p
                const float vp[3] = {vx, vy, vz}, mu[3] = {m0, m1, m2};
                const float vS[9] = {vSc00, vSc01, vSc02, vSc01, vSc11, vSc12, vSc02, vSc12, vSc22};
                float* ps = pose_s + threadIdx.x;
#pragma unroll
                for (int i = 0; i < 3; ++i) {
#pragma unroll
                    for (int j = 0; j < 3; ++j)
                        ps[(i * 3 + j) * kProjBwdThreads] = vp[i] * mu[j] + 2.0f * (vS[i * 3] * A[j] + vS[i * 3 + 1] * A[3 + j] + vS[i * 3 + 2] * A[6 + j]);
                    ps[(9 + i) * kProjBwdThreads] = vp[i];
                }
            }
            // ---- back to world: v_mu = W^T v_p ; vSigma = W^T vSc W ----
            vm0 += W[0] * vx + W[3] * vy + W[6] * vz;
            vm1 += W[1] * vx + W[4] * vy + W[7] * vz;
            vm2 += W[2] * vx + W[5] * vy + W[8] * vz;
            // T = vSc W (3x3), vSc symmetric
            float T[9];
            for (int j = 0; j < 3; ++j) {
                T[0 * 3 + j] = vSc00 * W[0 + j] + vSc01 * W[3 + j] + vSc02 * W[6 + j];
                T[1 * 3 + j] = vSc01 * W[0 + j] + vSc11 * W[3 + j] + vSc12 * W[6 + j];
                T[2 * 3 + j] = vSc02 * W[0 + j] + vSc12 * W[3 + j] + vSc22 * W[6 + j];
            }
            vS00 += W[0] * T[0] + W[3] * T[3] + W[6] * T[6];
            vS01 += W[0] * T[1] + W[3] * T[4] + W[6] * T[7];
            vS02 += W[0] * T[2] + W[3] * T[5] + W[6] * T[8];
            vS11 += W[1] * T[1] + W[4] * T[4] + W[7] * T[7];
            vS12 += W[1] * T[2] + W[4] * T[5] + W[7] * T[8];
            vS22 += W[2] * T[2] + W[5] * T[5] + W[8] * T[8];

            // ---- colour ----
            if (p.n_color > 0) {
                if (DEG < 0) {
                    float* dst = p.v_colors_in + (p.colors_per_camera ? idx * 3 : (int64_t)n * 3);
                    if (p.colors_per_camera) {
                        dst[0] = g_col[0];
                        dst[1] = g_col[1];
                        dst[2] = g_col[2];
                    } else {  // own row: accumulate over cameras (row zeroed below before the loop)
                        dst[0] += g_col[0];
                        dst[1] += g_col[1];
                        dst[2] += g_col[2];
                    }
                } else {
                    float dx = m0 - cam.campos[0], dy = m1 - cam.campos[1], dz = m2 - cam.campos[2];
                    float dn = fmaxf(sqrtf(dx * dx + dy * dy + dz * dz), 1e-12f);
                    const float rdn = 1.0f / dn;
                    float ux = dx * rdn, uy = dy * rdn, uz = dz * rdn;
                    float b[16], vb[16];
                    sh_bases_b<DG>(ux, uy, uz, b);
#pragma unroll
                    for (int k = 0; k < 16; ++k) vb[k] = 0.0f;
                    // pre-clamp colour to gate the gradient
                    float pre[3] = {0, 0, 0};
                    if (VEC) {
#pragma unroll
                        for (int j = 0; j < Sh::kVec; ++j) {
                            float4 cf = my_coef[j];
                            float cfa[4] = {cf.x, cf.y, cf.z, cf.w};
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int f = 4 * j + i;
                                if (f < Sh::kFloats) pre[f % 3] += b[f / 3] * cfa[i];
                            }
                        }
                    } else {
                        const float* row = p.colors_in + (int64_t)n * row_floats;
                        for (int f = 0; f < Sh::kFloats; ++f) pre[f % 3] += b[f / 3] * row[f];
                    }
                    float vpre[3];
#pragma unroll
                    for (int ch = 0; ch < 3; ++ch) vpre[ch] = (pre[ch] + 0.5f >= 0.0f) ? g_col[ch] : 0.0f;
                    if (VEC && XCH) {
                        // the coefficient gradient b (x) vpre is rebuilt on every rank from the exchanged colour gradients
                        // (qed_sh_grad_from_view_colors); only the direction term needs the coefficients here
#pragma unroll
                        for (int j = 0; j < Sh::kVec; ++j) {
                            float4 cf = my_coef[j];
                            float cfa[4] = {cf.x, cf.y, cf.z, cf.w};
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int f = 4 * j + i;
                                if (f < Sh::kFloats) vb[f / 3] += cfa[i] * vpre[f % 3];
                            }
                        }
                        xch_store(p, (int64_t)(p.xch_slot0 + c) * p.N + n, make_float4(vpre[0], vpre[1], vpre[2], p.xch_tag));
                    } else if (VEC) {
#pragma unroll
                        for (int j = 0; j < Sh::kVec; ++j) {
                            float4 cf = my_coef[j];
                            float cfa[4] = {cf.x, cf.y, cf.z, cf.w};
                            float out[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                            if (!ONE) {
                                const float4 acc = my_vcoef[j];
                                out[0] = acc.x;
                                out[1] = acc.y;
                                out[2] = acc.z;
                                out[3] = acc.w;
                            }
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int f = 4 * j + i;
                                if (f < Sh::kFloats) {
                                    vb[f / 3] += cfa[i] * vpre[f % 3];
                                    out[i] += b[f / 3] * vpre[f % 3];
                                }
                            }
                            my_vcoef[j] = make_float4(out[0], out[1], out[2], out[3]);
                        }
                    } else {
                        const float* row = p.colors_in + (int64_t)n * row_floats;
                        float* vrow = p.v_colors_in + (int64_t)n * row_floats;
                        for (int f = 0; f < Sh::kFloats; ++f) {
                            vb[f / 3] += row[f] * vpre[f % 3];
                            vrow[f] += b[f / 3] * vpre[f % 3];
                        }
                    }
                    float vux, vuy, vuz;
                    sh_bases_vjp<DG>(ux, uy, uz, vb, vux, vuy, vuz);
                    float dotp = vux * ux + vuy * uy + vuz * uz;
                    const float vdx = (vux - dotp * ux) * rdn, vdy = (vuy - dotp * uy) * rdn, vdz = (vuz - dotp * uz) * rdn;
                    vm0 += vdx;
                    vm1 += vdy;
                    vm2 += vdz;
                    if (POSE) {  // d = mu - campos: the view's campos gets -sum v_d (pose_finish_kernel)
                        pose_s[12 * kProjBwdThreads + threadIdx.x] = vdx;
                        pose_s[13 * kProjBwdThreads + threadIdx.x] = vdy;
                        pose_s[14 * kProjBwdThreads + threadIdx.x] = vdz;
                    }
                }
            }
        }
    }
    if (POSE) pose_flush(p, nC - 1, pose_s);  // ONE: the only view; else the last one

    if (in_range) {
        // ---- Sigma = M M^T ; M = R diag(s) ----
        // vM = 2 vSigma M  (vSigma symmetric)
        float R[9], M[9];
        quat_to_rotmat(qw, qx, qy, qz, R);
        for (int i = 0; i < 3; ++i) {
            M[i * 3 + 0] = R[i * 3 + 0] * s0;
            M[i * 3 + 1] = R[i * 3 + 1] * s1;
            M[i * 3 + 2] = R[i * 3 + 2] * s2;
        }
        float vM[9];
        for (int j = 0; j < 3; ++j) {
            vM[0 + j] = 2.0f * (vS00 * M[0 + j] + vS01 * M[3 + j] + vS02 * M[6 + j]);
            vM[3 + j] = 2.0f * (vS01 * M[0 + j] + vS11 * M[3 + j] + vS12 * M[6 + j]);
            vM[6 + j] = 2.0f * (vS02 * M[0 + j] + vS12 * M[3 + j] + vS22 * M[6 + j]);
        }
        float vs0 = R[0] * vM[0] + R[3] * vM[3] + R[6] * vM[6];
        float vs1 = R[1] * vM[1] + R[4] * vM[4] + R[7] * vM[7];
        float vs2 = R[2] * vM[2] + R[5] * vM[5] + R[8] * vM[8];
        float vR[9];
        for (int i = 0; i < 3; ++i) {
            vR[i * 3 + 0] = vM[i * 3 + 0] * s0;
            vR[i * 3 + 1] = vM[i * 3 + 1] * s1;
            vR[i * 3 + 2] = vM[i * 3 + 2] * s2;
        }
        float vw = 2.0f * (qz * (vR[3] - vR[1]) + qy * (vR[2] - vR[6]) + qx * (vR[7] - vR[5]));
        float vx = 2.0f * (qy * (vR[1] + vR[3]) + qz * (vR[2] + vR[6]) + qw * (vR[7] - vR[5]) - 2.0f * qx * (vR[4] + vR[8]));
        float vy = 2.0f * (qx * (vR[1] + vR[3]) + qz * (vR[5] + vR[7]) + qw * (vR[2] - vR[6]) - 2.0f * qy * (vR[0] + vR[8]));
        float vz = 2.0f * (qx * (vR[2] + vR[6]) + qy * (vR[5] + vR[7]) + qw * (vR[3] - vR[1]) - 2.0f * qz * (vR[0] + vR[4]));
        float dotq = vw * qw + vx * qx + vy * qy + vz * qz;
        const float rqn = 1.0f / qn;
        float4 vq = make_float4((vw - dotq * qw) * rqn, (vx - dotq * qx) * rqn, (vy - dotq * qy) * rqn, (vz - dotq * qz) * rqn);
        p.v_means[n * 3 + 0] = vm0;
        p.v_means[n * 3 + 1] = vm1;
        p.v_means[n * 3 + 2] = vm2;
        float* vqp = p.v_quats + (int64_t)n * 4;
        vqp[0] = vq.x;
        vqp[1] = vq.y;
        vqp[2] = vq.z;
        vqp[3] = vq.w;
        if (p.activations & QED_ACT_LOG_SCALES) {  // d/d log s = s d/ds
            vs0 *= s0;
            vs1 *= s1;
            vs2 *= s2;
        }
        if (p.activations & QED_ACT_LOGIT_OPACITIES) vopac *= opac * (1.0f - opac);  // sigmoid'
        p.v_scales[n * 3 + 0] = vs0;
        p.v_scales[n * 3 + 1] = vs1;
        p.v_scales[n * 3 + 2] = vs2;
        if (p.v_opacities) p.v_opacities[n] = vopac;
    }

    // ---- camera positions of this rank's views, for the ranks that rebuild the coefficient gradient ----
    if (XCH && blockIdx.x == 0 && threadIdx.x < p.C) {
        const CamB& cam = cams[threadIdx.x];
        xch_store(p, (int64_t)p.xch_total_slots * p.N + p.xch_slot0 + threadIdx.x, make_float4(cam.campos[0], cam.campos[1], cam.campos[2], p.xch_tag));
    }

    // ---- stream the coefficient gradient out (all K rows; unused ones are zero) ----
    if (use_sh && VEC && !XCH) {
        __syncwarp();
        const int64_t row0 = (int64_t)blockIdx.x * kProjBwdThreads + warp * 32;
        const int row_vec = row_floats / 4;
        float4* dst = reinterpret_cast<float4*>(p.v_colors_in) + row0 * row_vec;
        const float4* wbuf = vcoefbuf + warp * 32 * Sh::kStrideVec;
        const int rows = (p.N - row0) < 32 ? (int)(p.N - row0) : 32;
        if (Sh::kVec == 12 && row_vec == 12) {  // same lane -> (row, column) mapping as the staging above
            const int r0 = lane >> 2, j0 = lane & 3;
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
                const int r = r0 + 8 * rr;
                if (r < rows) {
#pragma unroll
                    for (int jj = 0; jj < 3; ++jj) dst[r * 12 + j0 + 4 * jj] = wbuf[r * Sh::kStrideVec + j0 + 4 * jj];
                }
            }
        } else {
            for (int q = lane; q < rows * row_vec; q += 32) {
                int r = q / row_vec, j = q - r * row_vec;
                float4 v = (j < Sh::kVec) ? wbuf[r * Sh::kStrideVec + j] : make_float4(0, 0, 0, 0);
                dst[q] = v;
            }
        }
    }
}

template <int DEG, bool VEC, bool XCH = false, int ONE = 0, bool POSE = false>
static int launch_project_bwd(const ProjBwdParams& p, cudaStream_t stream) {
    using Sh = ShShapeB<(DEG < 0 ? 0 : DEG)>;
    size_t smem = (size_t)p.C * kCamFloatsB * 4 + (POSE ? (size_t)kPoseVals * kProjBwdThreads * 4 : 0);
    if (DEG >= 0 && p.n_color > 0) smem += (size_t)((XCH || ONE) ? 1 : 2) * kProjBwdThreads * Sh::kStrideVec * 16;
    auto kern = project_bwd_kernel<DEG, VEC, XCH, ONE, POSE>;
    if (smem > 48 * 1024) QED_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int blocks = (p.N + kProjBwdThreads - 1) / kProjBwdThreads;
    QED_CUDA_TRY(launch_pdl(kern, dim3(blocks), dim3(kProjBwdThreads), smem, stream, p));
    return QED_OK;
}

// ------------------------------------------------------------------------------------------------
// Pose gradient, second pass: one block per view sums the per-warp partials of project_bwd_kernel<POSE> in a fixed order
// (float64), then applies the camera-position term of the SH direction.  campos = -W^-1 t with the GENERAL inverse (what
// the oracle's adjugate form and gsplat differentiate; it equals W^T only for an exactly orthonormal W), d = mu - campos:
//   g = W^-T sum_n v_d,   v_t += g,   v_W += g campos^T.
// v_viewmats[c] is overwritten; its row 3 is zero.
// ------------------------------------------------------------------------------------------------
constexpr int kPoseFinishThreads = 256;

__global__ void __launch_bounds__(kPoseFinishThreads) pose_finish_kernel(int warps, const float4* __restrict__ ws,
                                                                         const float* __restrict__ viewmats, float* __restrict__ v_viewmats) {
    __shared__ double part[kPoseFinishThreads / 32][kPoseVals];
    pdl_enter();
    const int c = blockIdx.x;
    double acc[kPoseVals];
#pragma unroll
    for (int k = 0; k < kPoseVals; ++k) acc[k] = 0.0;
    for (int w = threadIdx.x; w < warps; w += kPoseFinishThreads) {
        const float4* r = ws + ((int64_t)c * warps + w) * 4;
        const float4 a = r[0], b = r[1], d = r[2], e = r[3];
        const float v[kPoseVals] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, d.x, d.y, d.z, d.w, e.x, e.y, e.z};
#pragma unroll
        for (int k = 0; k < kPoseVals; ++k) acc[k] += (double)v[k];
    }
#pragma unroll
    for (int k = 0; k < kPoseVals; ++k) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], off);
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < kPoseVals; ++k) part[threadIdx.x >> 5][k] = acc[k];
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    double s[kPoseVals];
    for (int k = 0; k < kPoseVals; ++k) {
        s[k] = part[0][k];
        for (int w = 1; w < kPoseFinishThreads / 32; ++w) s[k] += part[w][k];
    }
    const float* V = viewmats + (int64_t)c * 16;
    double vW[9], vt[3];
    for (int k = 0; k < 9; ++k) vW[k] = s[k];
    for (int i = 0; i < 3; ++i) vt[i] = s[9 + i];
    if (s[12] != 0.0 || s[13] != 0.0 || s[14] != 0.0) {
        double a[3][3], t[3];
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) a[i][j] = V[i * 4 + j];
            t[i] = V[i * 4 + 3];
        }
        // inverse = adjugate / det, the cofactors of load_camera_b
        double inv[3][3];
        inv[0][0] = a[1][1] * a[2][2] - a[1][2] * a[2][1];
        inv[0][1] = a[0][2] * a[2][1] - a[0][1] * a[2][2];
        inv[0][2] = a[0][1] * a[1][2] - a[0][2] * a[1][1];
        inv[1][0] = a[1][2] * a[2][0] - a[1][0] * a[2][2];
        inv[1][1] = a[0][0] * a[2][2] - a[0][2] * a[2][0];
        inv[1][2] = a[0][2] * a[1][0] - a[0][0] * a[1][2];
        inv[2][0] = a[1][0] * a[2][1] - a[1][1] * a[2][0];
        inv[2][1] = a[0][1] * a[2][0] - a[0][0] * a[2][1];
        inv[2][2] = a[0][0] * a[1][1] - a[0][1] * a[1][0];
        const double rdet = 1.0 / (a[0][0] * inv[0][0] + a[0][1] * inv[1][0] + a[0][2] * inv[2][0]);
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) inv[i][j] *= rdet;
        double campos[3], g[3];
        for (int i = 0; i < 3; ++i) campos[i] = -(inv[i][0] * t[0] + inv[i][1] * t[1] + inv[i][2] * t[2]);
        for (int i = 0; i < 3; ++i) g[i] = inv[0][i] * s[12] + inv[1][i] * s[13] + inv[2][i] * s[14];  // W^-T sum v_d
        for (int i = 0; i < 3; ++i) {
            vt[i] += g[i];
            for (int j = 0; j < 3; ++j) vW[i * 3 + j] += g[i] * campos[j];
        }
    }
    float* out = v_viewmats + (int64_t)c * 16;
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) out[i * 4 + j] = (float)vW[i * 3 + j];
        out[i * 4 + 3] = (float)vt[i];
    }
    for (int j = 12; j < 16; ++j) out[j] = 0.0f;
}

// bytes of the per-warp partials of qed_project_bwd_pose
static size_t pose_workspace_bytes(int C, int N) {
    if (C <= 0 || N <= 0) return 0;
    const size_t warps = (size_t)((N + kProjBwdThreads - 1) / kProjBwdThreads) * (kProjBwdThreads / 32);
    return (size_t)C * warps * 4 * sizeof(float4);
}

// ------------------------------------------------------------------------------------------------
// SH coefficient gradient rebuilt from exchanged per-view colour gradients (multi-GPU, see qed_project_bwd_exchange).
// d colour / d coeff[k, ch] = basis_k(direction) for every view, so   v_sh[n] = sum_views  basis(dir(n, view)) (x) v_colour(n, view):
// rank-1 per view.  Every rank evaluates the sum over ALL views of the batch, in view order, from the same bits --
// replicas stay bit-identical -- and 16 B per visible (view, Gaussian) cross NVLink instead of a 192-B row per Gaussian
// through an all-reduce.  One thread per Gaussian, 48 accumulators in registers, rows streamed out through shared
// memory with coalesced 16-byte stores (the pattern of project_bwd_kernel).
// ------------------------------------------------------------------------------------------------
constexpr int kShGradThreads = 128;

template <int DEG>
__global__ void __launch_bounds__(kShGradThreads) sh_grad_from_view_colors_kernel(int V, int N, int K, const float* __restrict__ means,
                                                                                 const float4* __restrict__ xch, float tag,
                                                                                 float* __restrict__ v_sh) {
    using Sh = ShShapeB<DEG>;
    extern __shared__ float4 smem4[];
    pdl_enter();
    float4* rows = smem4;  // [kShGradThreads][kStrideVec]
    const int n = blockIdx.x * kShGradThreads + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float4* campos = xch + (int64_t)V * N;
    float acc[Sh::kBases][3];
#pragma unroll
    for (int k = 0; k < Sh::kBases; ++k) acc[k][0] = acc[k][1] = acc[k][2] = 0.0f;
    if (n < N) {
        const float m0 = means[n * 3 + 0], m1 = means[n * 3 + 1], m2 = means[n * 3 + 2];
        for (int v0 = 0; v0 < V; v0 += 4) {  // four views' records in flight per thread
            float4 vc[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) vc[u] = (v0 + u < V) ? xch[(int64_t)(v0 + u) * N + n] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (v0 + u >= V || vc[u].w != tag) continue;  // not visible in that view this step (stale record)
                const float4 cp = campos[v0 + u];
                const float dx = m0 - cp.x, dy = m1 - cp.y, dz = m2 - cp.z;
                const float dn = fmaxf(sqrtf(dx * dx + dy * dy + dz * dz), 1e-12f);
                float b[16];
                sh_bases_b<DEG>(dx / dn, dy / dn, dz / dn, b);
#pragma unroll
                for (int k = 0; k < Sh::kBases; ++k) {
                    acc[k][0] = fmaf(b[k], vc[u].x, acc[k][0]);
                    acc[k][1] = fmaf(b[k], vc[u].y, acc[k][1]);
                    acc[k][2] = fmaf(b[k], vc[u].z, acc[k][2]);
                }
            }
        }
    }
    float* my = reinterpret_cast<float*>(rows + (warp * 32 + lane) * Sh::kStrideVec);
#pragma unroll
    for (int k = 0; k < Sh::kBases; ++k) {
        my[k * 3 + 0] = acc[k][0];
        my[k * 3 + 1] = acc[k][1];
        my[k * 3 + 2] = acc[k][2];
    }
#pragma unroll
    for (int f = Sh::kFloats; f < Sh::kVec * 4; ++f) my[f] = 0.0f;
    __syncwarp();
    const int64_t row0 = (int64_t)blockIdx.x * kShGradThreads + warp * 32;
    const int row_vec = K * 3 / 4;
    float4* dst = reinterpret_cast<float4*>(v_sh) + row0 * row_vec;
    const float4* wbuf = rows + warp * 32 * Sh::kStrideVec;
    const int nrows = (N - row0) < 32 ? (int)(N - row0) : 32;
    for (int q = lane; q < nrows * row_vec; q += 32) {
        const int r = q / row_vec, j = q - r * row_vec;
        dst[q] = (j < Sh::kVec) ? wbuf[r * Sh::kStrideVec + j] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

template <int DEG>
static int launch_sh_grad(int V, int N, int K, const float* means, const float4* xch, float tag, float* v_sh, cudaStream_t stream) {
    using Sh = ShShapeB<DEG>;
    const size_t smem = (size_t)kShGradThreads * Sh::kStrideVec * 16;
    QED_CUDA_TRY(launch_pdl(sh_grad_from_view_colors_kernel<DEG>, dim3((N + kShGradThreads - 1) / kShGradThreads), dim3(kShGradThreads), smem, stream, V, N,
                            K, means, xch, tag, v_sh));
    return QED_OK;
}

}  // namespace qed

using namespace qed;

// test hook (thread-local): 0 = the single-view specialisation of the projection backward is not used
static thread_local int g_projbwd_one = 5;
extern "C" int qed_debug_set_project_bwd_one(int blocks) {  // 0 = off, 5 / 6 = resident blocks per SM of the specialisation
    int old = g_projbwd_one;
    g_projbwd_one = (blocks == 6) ? 6 : (blocks ? 5 : 0);
    return old;
}

template <bool POSE>
static int dispatch_project_bwd(const ProjBwdParams& p, bool vec_ok, cudaStream_t stream) {
    switch (p.sh_degree) {
        case 0: return vec_ok ? launch_project_bwd<0, true, false, 0, POSE>(p, stream) : launch_project_bwd<0, false, false, 0, POSE>(p, stream);
        case 1: return vec_ok ? launch_project_bwd<1, true, false, 0, POSE>(p, stream) : launch_project_bwd<1, false, false, 0, POSE>(p, stream);
        case 2: return vec_ok ? launch_project_bwd<2, true, false, 0, POSE>(p, stream) : launch_project_bwd<2, false, false, 0, POSE>(p, stream);
        case 3:
            if constexpr (POSE) {  // 4 resident blocks (128 registers): at 5 or 6 the pose variant spills
                if (vec_ok && p.C == 1 && g_projbwd_one) return launch_project_bwd<3, true, false, 4, true>(p, stream);
            } else {
                if (vec_ok && p.C == 1 && g_projbwd_one == 6) return launch_project_bwd<3, true, false, 6>(p, stream);
                if (vec_ok && p.C == 1 && g_projbwd_one) return launch_project_bwd<3, true, false, 5>(p, stream);
            }
            return vec_ok ? launch_project_bwd<3, true, false, 0, POSE>(p, stream) : launch_project_bwd<3, false, false, 0, POSE>(p, stream);
        default: return launch_project_bwd<-1, false, false, 0, POSE>(p, stream);
    }
}

// v_viewmats != NULL: the POSE variant, with pose_ws = pose_workspace_bytes(C, N) of per-warp partials
static int project_bwd_impl(int C, int N, const float* means, const float* quats, const float* scales,
                            const float* opacities, int activations, const float* colors_in, int K, int sh_degree,
                            int colors_per_camera, const float* viewmats, const float* Ks, int width, int height,
                            float eps2d, int calc_compensations, int n_color, int append_depth,
                            const int32_t* radii, const float* conics, const float* compensations,
                            const float* v_means2d, const float* v_depths, const float* v_conics,
                            const float* v_colors, const float* v_opacities_cn, const float* packed_grads,
                            float* v_means, float* v_quats, float* v_scales, float* v_opacities,
                            float* v_colors_in, const ProjBwdParams* xch, float* v_viewmats, float4* pose_ws,
                            cudaStream_t stream) {
    if (C < 0 || N < 0) return QED_ERR_BAD_ARG;
    if (!(n_color == 0 || n_color == 3) || !(append_depth == 0 || append_depth == 1)) return QED_ERR_BAD_ARG;
    if (v_viewmats && C > 0 && N == 0) QED_CUDA_TRY(cudaMemsetAsync(v_viewmats, 0, (size_t)C * 16 * sizeof(float), stream));
    if (C == 0 || N == 0) return QED_OK;
    if (v_viewmats && !pose_ws) return QED_ERR_BAD_ARG;
    if (C > 1024) return QED_ERR_UNSUPPORTED;
    if (!means || !quats || !scales || !viewmats || !Ks || !radii || !conics || !v_means || !v_quats || !v_scales)
        return QED_ERR_BAD_ARG;
    if (calc_compensations && (!compensations || !opacities)) return QED_ERR_BAD_ARG;
    if (n_color > 0 && (!colors_in || (!v_colors_in && !xch))) return QED_ERR_BAD_ARG;
    if (n_color == 0) sh_degree = -1;
    if (sh_degree > 3) return QED_ERR_UNSUPPORTED;

    ProjBwdParams p{};
    if (xch) p = *xch;
    p.C = C;
    p.N = N;
    p.K = K;
    p.sh_degree = sh_degree;
    p.colors_per_camera = colors_per_camera;
    p.width = width;
    p.height = height;
    p.eps2d = eps2d;
    p.calc_comp = calc_compensations;
    p.activations = activations;
    p.n_color = n_color;
    p.append_depth = append_depth;
    p.means = means;
    p.quats = quats;
    p.scales = scales;
    p.opacities = opacities;
    p.colors_in = colors_in;
    p.viewmats = viewmats;
    p.Ks = Ks;
    p.radii = radii;
    p.conics = conics;
    p.comps = compensations;
    p.v_means2d = v_means2d;
    p.v_depths = v_depths;
    p.v_conics = v_conics;
    p.v_colors = v_colors;
    p.v_opac_cn = v_opacities_cn;
    p.packed = packed_grads;
    p.v_means = v_means;
    p.v_quats = v_quats;
    p.v_scales = v_scales;
    p.v_opacities = v_opacities;
    p.v_colors_in = v_colors_in;

    const bool vec_ok = sh_degree >= 0 && ((K * 3) % 4 == 0) && ((reinterpret_cast<uintptr_t>(colors_in) & 15) == 0) &&
                        (xch || (reinterpret_cast<uintptr_t>(v_colors_in) & 15) == 0);
    const auto pose_finish = [&]() -> int {
        const int warps = ((N + kProjBwdThreads - 1) / kProjBwdThreads) * (kProjBwdThreads / 32);
        QED_CUDA_TRY(launch_pdl(pose_finish_kernel, dim3(C), dim3(kPoseFinishThreads), 0, stream, warps, (const float4*)pose_ws, viewmats, v_viewmats));
        return QED_OK;
    };
    if (xch) {
        if (!vec_ok || n_color != 3) return QED_ERR_UNSUPPORTED;  // the exchange carries SH colour gradients
        if (!v_viewmats) {
            switch (sh_degree) {
                case 0: return launch_project_bwd<0, true, true>(p, stream);
                case 1: return launch_project_bwd<1, true, true>(p, stream);
                case 2: return launch_project_bwd<2, true, true>(p, stream);
                default: return launch_project_bwd<3, true, true>(p, stream);
            }
        }
        p.pose_ws = pose_ws;
        int rc;
        switch (sh_degree) {
            case 0: rc = launch_project_bwd<0, true, true, 0, true>(p, stream); break;
            case 1: rc = launch_project_bwd<1, true, true, 0, true>(p, stream); break;
            case 2: rc = launch_project_bwd<2, true, true, 0, true>(p, stream); break;
            default: rc = launch_project_bwd<3, true, true, 0, true>(p, stream); break;
        }
        return rc != QED_OK ? rc : pose_finish();
    }
    if (n_color > 0 && (sh_degree < 0 || !vec_ok)) {
        // fallback paths accumulate straight into v_colors_in: clear it first
        size_t bytes = sh_degree < 0 ? (size_t)(colors_per_camera ? (size_t)C * N : (size_t)N) * 3 * 4 : (size_t)N * K * 3 * 4;
        QED_CUDA_TRY(cudaMemsetAsync(v_colors_in, 0, bytes, stream));
    }
    if (!v_viewmats) return dispatch_project_bwd<false>(p, vec_ok, stream);
    p.pose_ws = pose_ws;
    const int rc = dispatch_project_bwd<true>(p, vec_ok, stream);
    return rc != QED_OK ? rc : pose_finish();
}

extern "C" int qed_project_bwd(int C, int N, const float* means, const float* quats, const float* scales,
                               const float* opacities, int activations, const float* colors_in, int K, int sh_degree,
                               int colors_per_camera, const float* viewmats, const float* Ks, int width, int height,
                               float eps2d, int calc_compensations, int n_color, int append_depth,
                               const int32_t* radii, const float* conics, const float* compensations,
                               const float* v_means2d, const float* v_depths, const float* v_conics,
                               const float* v_colors, const float* v_opacities_cn, const float* packed_grads,
                               float* v_means, float* v_quats, float* v_scales, float* v_opacities,
                               float* v_colors_in, qed_stream_t stream_) {
    return project_bwd_impl(C, N, means, quats, scales, opacities, activations, colors_in, K, sh_degree, colors_per_camera, viewmats, Ks, width,
                            height, eps2d, calc_compensations, n_color, append_depth, radii, conics, compensations, v_means2d, v_depths, v_conics,
                            v_colors, v_opacities_cn, packed_grads, v_means, v_quats, v_scales, v_opacities, v_colors_in, nullptr,
                            nullptr, nullptr, (cudaStream_t)stream_);
}

extern "C" size_t qed_project_bwd_pose_workspace_bytes(int C, int N) { return pose_workspace_bytes(C, N); }

extern "C" int qed_project_bwd_pose(int C, int N, const float* means, const float* quats, const float* scales,
                                    const float* opacities, int activations, const float* colors_in, int K, int sh_degree,
                                    int colors_per_camera, const float* viewmats, const float* Ks, int width, int height,
                                    float eps2d, int calc_compensations, int n_color, int append_depth,
                                    const int32_t* radii, const float* conics, const float* compensations,
                                    const float* v_means2d, const float* v_depths, const float* v_conics,
                                    const float* v_colors, const float* v_opacities_cn, const float* packed_grads,
                                    float* v_means, float* v_quats, float* v_scales, float* v_opacities,
                                    float* v_colors_in, float* v_viewmats, void* workspace, size_t workspace_bytes,
                                    qed_stream_t stream_) {
    if (C < 0 || N < 0) return QED_ERR_BAD_ARG;
    if (C == 0) return QED_OK;
    if (!v_viewmats) return QED_ERR_BAD_ARG;
    if (N > 0) {
        if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 15)) return QED_ERR_BAD_ARG;
        if (workspace_bytes < pose_workspace_bytes(C, N)) return QED_ERR_WORKSPACE;
    }
    return project_bwd_impl(C, N, means, quats, scales, opacities, activations, colors_in, K, sh_degree, colors_per_camera, viewmats, Ks, width,
                            height, eps2d, calc_compensations, n_color, append_depth, radii, conics, compensations, v_means2d, v_depths, v_conics,
                            v_colors, v_opacities_cn, packed_grads, v_means, v_quats, v_scales, v_opacities, v_colors_in, nullptr,
                            v_viewmats, reinterpret_cast<float4*>(workspace), (cudaStream_t)stream_);
}

static int project_bwd_exchange(int C, int N, const float* means, const float* quats, const float* scales, const float* opacities,
                                int activations, const float* sh_coeffs, int K, int sh_degree, const float* viewmats, const float* Ks, int width,
                                int height, float eps2d, int calc_compensations, int append_depth, const int32_t* radii, const float* conics,
                                const float* compensations, const float* packed_grads, float* v_means, float* v_quats, float* v_scales,
                                float* v_opacities, float* exchange_multicast, float* const* exchange_peers, int world, int first_slot,
                                int total_slots, float tag, float* v_viewmats, float4* pose_ws, cudaStream_t stream) {
    if (world < 1 || world > 16 || first_slot < 0 || C < 0 || first_slot + C > total_slots) return QED_ERR_BAD_ARG;
    if (!exchange_multicast && !exchange_peers) return QED_ERR_BAD_ARG;
    if (!packed_grads || sh_degree < 0) return QED_ERR_BAD_ARG;
    ProjBwdParams x{};
    x.xch_mc = reinterpret_cast<float4*>(exchange_multicast);
    for (int r = 0; r < world; ++r) {
        x.xch_peer[r] = exchange_peers ? reinterpret_cast<float4*>(exchange_peers[r]) : nullptr;
        if (!x.xch_mc && !x.xch_peer[r]) return QED_ERR_BAD_ARG;
    }
    x.xch_world = world;
    x.xch_slot0 = first_slot;
    x.xch_total_slots = total_slots;
    x.xch_tag = tag;
    return project_bwd_impl(C, N, means, quats, scales, opacities, activations, sh_coeffs, K, sh_degree, 0, viewmats, Ks, width, height, eps2d,
                            calc_compensations, 3, append_depth, radii, conics, compensations, nullptr, nullptr, nullptr, nullptr, nullptr,
                            packed_grads, v_means, v_quats, v_scales, v_opacities, nullptr, &x, v_viewmats, pose_ws, stream);
}

extern "C" int qed_project_bwd_exchange(int C, int N, const float* means, const float* quats, const float* scales,
                                        const float* opacities, int activations, const float* sh_coeffs, int K, int sh_degree,
                                        const float* viewmats, const float* Ks, int width, int height, float eps2d,
                                        int calc_compensations, int append_depth, const int32_t* radii, const float* conics,
                                        const float* compensations, const float* packed_grads, float* v_means, float* v_quats,
                                        float* v_scales, float* v_opacities, float* exchange_multicast, float* const* exchange_peers,
                                        int world, int first_slot, int total_slots, float tag, qed_stream_t stream_) {
    return project_bwd_exchange(C, N, means, quats, scales, opacities, activations, sh_coeffs, K, sh_degree, viewmats, Ks, width, height, eps2d,
                                calc_compensations, append_depth, radii, conics, compensations, packed_grads, v_means, v_quats, v_scales,
                                v_opacities, exchange_multicast, exchange_peers, world, first_slot, total_slots, tag, nullptr, nullptr,
                                (cudaStream_t)stream_);
}

extern "C" int qed_project_bwd_exchange_pose(int C, int N, const float* means, const float* quats, const float* scales,
                                             const float* opacities, int activations, const float* sh_coeffs, int K, int sh_degree,
                                             const float* viewmats, const float* Ks, int width, int height, float eps2d,
                                             int calc_compensations, int append_depth, const int32_t* radii, const float* conics,
                                             const float* compensations, const float* packed_grads, float* v_means, float* v_quats,
                                             float* v_scales, float* v_opacities, float* exchange_multicast, float* const* exchange_peers,
                                             int world, int first_slot, int total_slots, float tag, float* v_viewmats, void* pose_ws,
                                             size_t ws_bytes, qed_stream_t stream_) {
    if (C < 0 || N < 0) return QED_ERR_BAD_ARG;
    if (C == 0) return QED_OK;
    if (!v_viewmats) return QED_ERR_BAD_ARG;
    if (N > 0) {
        if (!pose_ws || (reinterpret_cast<uintptr_t>(pose_ws) & 15)) return QED_ERR_BAD_ARG;
        if (ws_bytes < pose_workspace_bytes(C, N)) return QED_ERR_WORKSPACE;
    }
    return project_bwd_exchange(C, N, means, quats, scales, opacities, activations, sh_coeffs, K, sh_degree, viewmats, Ks, width, height, eps2d,
                                calc_compensations, append_depth, radii, conics, compensations, packed_grads, v_means, v_quats, v_scales,
                                v_opacities, exchange_multicast, exchange_peers, world, first_slot, total_slots, tag, v_viewmats,
                                reinterpret_cast<float4*>(pose_ws), (cudaStream_t)stream_);
}

extern "C" int qed_sh_grad_from_view_colors(int total_slots, int N, int K, int sh_degree, const float* means, const float* exchange_local,
                                            float tag, float* v_sh, qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (total_slots < 0 || N < 0 || K <= 0 || sh_degree < 0 || sh_degree > 3 || (sh_degree + 1) * (sh_degree + 1) > K) return QED_ERR_BAD_ARG;
    if (N == 0) return QED_OK;
    if (!means || !exchange_local || !v_sh) return QED_ERR_BAD_ARG;
    if ((K * 3) % 4 || (reinterpret_cast<uintptr_t>(v_sh) & 15) || (reinterpret_cast<uintptr_t>(exchange_local) & 15)) return QED_ERR_BAD_ARG;
    const float4* x = reinterpret_cast<const float4*>(exchange_local);
    switch (sh_degree) {
        case 0: return launch_sh_grad<0>(total_slots, N, K, means, x, tag, v_sh, stream);
        case 1: return launch_sh_grad<1>(total_slots, N, K, means, x, tag, v_sh, stream);
        case 2: return launch_sh_grad<2>(total_slots, N, K, means, x, tag, v_sh, stream);
        default: return launch_sh_grad<3>(total_slots, N, K, means, x, tag, v_sh, stream);
    }
}
