// (a1) camera-to-world -> gsplat world-to-camera, the `get_viewmat` of qed_splatter/model.py:22-38:
//   R = c2w[:, :3, :3] * [1, -1, -1]   (flip the y and z COLUMNS: nerfstudio/OpenGL -> gsplat/OpenCV camera axes)
//   viewmat = [[R^T, -R^T T], [0 0 0 1]]          (analytic inverse of a rigid transform)
// One thread per camera; every product and sum is an individually rounded IEEE operation in a fixed order
// (((r0 t0 + r1 t1) + r2 t2), negated), which is what oracle/torch_impl.py::get_viewmat's float32 bmm evaluates to on
// the host cores, so the result is bit-identical to the oracle (tests/test_gpu_data_side.py).
#include "common.cuh"

namespace qed {

// viewmat = [[R^T, -R^T T], [0 0 0 1]] for the column-flipped rotation R, in the pinned order above
__device__ __forceinline__ void write_viewmat(const float (&R)[3][3], const float (&T)[3], float* __restrict__ v) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {  // row i of R^T = column i of R
        v[i * 4 + 0] = R[0][i];
        v[i * 4 + 1] = R[1][i];
        v[i * 4 + 2] = R[2][i];
        v[i * 4 + 3] = -add(add(mul(R[0][i], T[0]), mul(R[1][i], T[1])), mul(R[2][i], T[2]));
    }
    v[12] = 0.0f;
    v[13] = 0.0f;
    v[14] = 0.0f;
    v[15] = 1.0f;
}

__global__ void viewmat_from_c2w_kernel(int C, int rows, const float* __restrict__ c2w, float* __restrict__ viewmats) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float* m = c2w + (int64_t)c * rows * 4;
    float R[3][3], T[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        R[i][0] = m[i * 4 + 0];
        R[i][1] = -m[i * 4 + 1];
        R[i][2] = -m[i * 4 + 2];
        T[i] = m[i * 4 + 3];
    }
    write_viewmat(R, T, viewmats + (int64_t)c * 16);
}

// Backward of viewmat_from_c2w_kernel.  Rf = c2w[:3,:3] diag(1,-1,-1), T = c2w[:3,3]; viewmat = [[Rf^T, -Rf^T T], [0 0 0 1]]:
//   v_Rf = v_rot^T - T v_trans^T,  v_T = -Rf v_trans,  v_c2w[:3,:3] = v_Rf diag(1,-1,-1),  v_c2w[:3,3] = v_T.
// Row 3 of v_viewmats is ignored (constant); row 3 of a [C,4,4] c2w gets zero.
__global__ void viewmat_from_c2w_bwd_kernel(int C, int rows, const float* __restrict__ c2w, const float* __restrict__ v_viewmats,
                                            float* __restrict__ v_c2w) {
    pdl_enter();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float* m = c2w + (int64_t)c * rows * 4;
    const float* g = v_viewmats + (int64_t)c * 16;
    float* out = v_c2w + (int64_t)c * rows * 4;
    const float sgn[3] = {1.0f, -1.0f, -1.0f};
    float Rf[3][3], T[3], vtr[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) Rf[i][j] = sgn[j] * m[i * 4 + j];
        T[i] = m[i * 4 + 3];
        vtr[i] = g[i * 4 + 3];
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) out[i * 4 + j] = sgn[j] * (g[j * 4 + i] - T[i] * vtr[j]);  // v_Rf[i][j] = v_rot[j][i] - T_i v_trans_j
        out[i * 4 + 3] = -(Rf[i][0] * vtr[0] + Rf[i][1] * vtr[1] + Rf[i][2] * vtr[2]);
    }
    if (rows == 4) {
#pragma unroll
        for (int j = 12; j < 16; ++j) out[j] = 0.0f;
    }
}

// ------------------------------------------------------------------------------------------------
// (a1') splatfacto's camera optimizer, mode SO3xR3 (nerfstudio CameraOptimizer.apply_to_camera, model.py:212/246).
// A table pose_adjustment[num_cameras, 6] = {t (3), omega (3)}; view c uses row camera_ids[c]:
//   theta^2 = max(|omega|^2, 1e-4),  R = I + (sin theta / theta) [omega]x + ((1 - cos theta) / theta^2) [omega]x^2
//   c2w' = c2w[:3,:4] @ [[R, t], [0, 1]]:  R' = Rc R,  t' = Rc t + tc  (SO3 x R3: t is not rotated)
//   viewmat = get_viewmat(c2w')
// ------------------------------------------------------------------------------------------------

struct SO3Exp {
    double K[3][3];  // [omega]x
    double S[3][3];  // R - I = A K + B K^2
    double A, B, theta, w[3];
    bool clamped;    // |omega|^2 < 1e-4: theta is the constant 0.01, A and B do not depend on omega
};

__device__ __forceinline__ void so3_exp(const float* __restrict__ a, SO3Exp& e) {
    for (int i = 0; i < 3; ++i) e.w[i] = a[3 + i];
    const double n2 = e.w[0] * e.w[0] + e.w[1] * e.w[1] + e.w[2] * e.w[2];
    e.clamped = !(n2 >= 1e-4);  // torch.clamp passes the gradient at the bound itself
    const double th2 = e.clamped ? 1e-4 : n2;
    e.theta = sqrt(th2);
    e.A = sin(e.theta) / e.theta;
    e.B = (1.0 - cos(e.theta)) / th2;
    const double* w = e.w;
    const double K[3][3] = {{0.0, -w[2], w[1]}, {w[2], 0.0, -w[0]}, {-w[1], w[0], 0.0}};
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            e.K[i][j] = K[i][j];
            const double K2 = w[i] * w[j] - (i == j ? n2 : 0.0);  // [omega]x^2 = omega omega^T - |omega|^2 I
            e.S[i][j] = e.A * K[i][j] + e.B * K2;
        }
}

// x + d rounded once, and x itself (all its bits, the sign of a zero too) when the correction is exactly zero: a zero
// table row then reproduces qed_viewmat_from_c2w bit for bit
__device__ __forceinline__ float plus_nz(float x, double d) { return d != 0.0 ? (float)((double)x + d) : x; }

__global__ void camera_opt_apply_kernel(int C, int rows, int num_cameras, const int32_t* __restrict__ camera_ids, const float* __restrict__ c2w,
                                        const float* __restrict__ adj, float* __restrict__ viewmats) {
    pdl_enter();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const int id = camera_ids[c];
    float* v = viewmats + (int64_t)c * 16;
    if (id < 0 || id >= num_cameras) {  // the host validates; never read outside the table
        for (int k = 0; k < 16; ++k) v[k] = __int_as_float(0x7fffffff);
        return;
    }
    const float* m = c2w + (int64_t)c * rows * 4;
    const float* a = adj + (int64_t)id * 6;
    SO3Exp e;
    so3_exp(a, e);
    float R[3][3], T[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double dt = 0.0;
        for (int k = 0; k < 3; ++k) dt += (double)m[i * 4 + k] * (double)a[k];
        T[i] = plus_nz(m[i * 4 + 3], dt);
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            double d = 0.0;
            for (int k = 0; k < 3; ++k) d += (double)m[i * 4 + k] * e.S[k][j];
            const float r = plus_nz(m[i * 4 + j], d);
            R[i][j] = j == 0 ? r : -r;
        }
    }
    write_viewmat(R, T, v);
}

// <M, [e_m]x> for m = 0, 1, 2
__device__ __forceinline__ void skew_dot(const double (&M)[3][3], double (&out)[3]) {
    out[0] = M[2][1] - M[1][2];
    out[1] = M[0][2] - M[2][0];
    out[2] = M[1][0] - M[0][1];
}

// One thread per table row: the views with that camera id, in view order, in float64 (no atomics, the same bits from
// call to call).  Per view: the viewmat backward of viewmat_from_c2w_bwd_kernel on c2w', v_R = Rc^T v_R', v_t = Rc^T v_t',
// then the VJP of the exp map.
__global__ void camera_opt_bwd_kernel(int C, int rows, int num_cameras, const int32_t* __restrict__ camera_ids, const float* __restrict__ c2w,
                                      const float* __restrict__ adj, const float* __restrict__ v_viewmats, float* __restrict__ v_adj) {
    pdl_enter();
    const int j0 = blockIdx.x * blockDim.x + threadIdx.x;
    if (j0 >= num_cameras) return;
    const float* a = adj + (int64_t)j0 * 6;
    SO3Exp e;
    so3_exp(a, e);
    double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    const double sgn[3] = {1.0, -1.0, -1.0};
    for (int c = 0; c < C; ++c) {
        if (camera_ids[c] != j0) continue;
        const float* m = c2w + (int64_t)c * rows * 4;
        const float* g = v_viewmats + (int64_t)c * 16;
        double Rc[3][3], Rp[3][3], tp[3], vtr[3];
        for (int i = 0; i < 3; ++i) {
            for (int k = 0; k < 3; ++k) Rc[i][k] = m[i * 4 + k];
            vtr[i] = g[i * 4 + 3];
        }
        for (int i = 0; i < 3; ++i) {
            tp[i] = (double)m[i * 4 + 3];
            for (int k = 0; k < 3; ++k) tp[i] += Rc[i][k] * (double)a[k];
            for (int j = 0; j < 3; ++j) {
                Rp[i][j] = Rc[i][j];
                for (int k = 0; k < 3; ++k) Rp[i][j] += Rc[i][k] * e.S[k][j];
            }
        }
        // viewmat = [[Rf^T, -Rf^T t'], ...], Rf = R' diag(sgn):  v_R'[i][j] = sgn_j (v_rot[j][i] - t'_i v_trans_j),  v_t' = -Rf v_trans
        double vRp[3][3], vtp[3];
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) vRp[i][j] = sgn[j] * ((double)g[j * 4 + i] - tp[i] * vtr[j]);
            vtp[i] = -(Rp[i][0] * vtr[0] - Rp[i][1] * vtr[1] - Rp[i][2] * vtr[2]);
        }
        double vR[3][3];
        for (int i = 0; i < 3; ++i) {
            double s = 0.0;
            for (int k = 0; k < 3; ++k) s += Rc[k][i] * vtp[k];
            acc[i] += s;
            for (int j = 0; j < 3; ++j) {
                double r = 0.0;
                for (int k = 0; k < 3; ++k) r += Rc[k][i] * vRp[k][j];
                vR[i][j] = r;
            }
        }
        // R = I + A K + B K^2:  d/d omega_m = A E_m + B (E_m K + K E_m) + (A' K + B' K^2) omega_m / theta  (A', B' = 0 when clamped)
        double vRKt[3][3], KtvR[3][3], dK = 0.0, dK2 = 0.0;
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                double x = 0.0, y = 0.0, k2 = 0.0;
                for (int k = 0; k < 3; ++k) {
                    x += vR[i][k] * e.K[j][k];
                    y += e.K[k][i] * vR[k][j];
                    k2 += e.K[i][k] * e.K[k][j];
                }
                vRKt[i][j] = x;
                KtvR[i][j] = y;
                dK += vR[i][j] * e.K[i][j];
                dK2 += vR[i][j] * k2;
            }
        double s0[3], s1[3], s2[3];
        skew_dot(vR, s0);
        skew_dot(vRKt, s1);
        skew_dot(KtvR, s2);
        double radial = 0.0;
        if (!e.clamped) {
            const double dA = (cos(e.theta) - e.A) / e.theta, dB = (e.A - 2.0 * e.B) / e.theta;
            radial = (dA * dK + dB * dK2) / e.theta;
        }
        for (int m3 = 0; m3 < 3; ++m3) acc[3 + m3] += e.A * s0[m3] + e.B * (s1[m3] + s2[m3]) + radial * e.w[m3];
    }
    float* out = v_adj + (int64_t)j0 * 6;
    for (int k = 0; k < 6; ++k) out[k] = (float)acc[k];
}

// Regulariser of CameraOptimizer.get_loss_dict: trans_weight * mean_rows |t| + rot_weight * mean_rows |omega| over all rows.
// One block; fixed-order float64 sums.  Its gradient (zero at a zero norm, as in torch) is ADDED to v_adj.
constexpr int kCamRegThreads = 256;

__global__ void __launch_bounds__(kCamRegThreads) camera_opt_reg_kernel(int num_cameras, const float* __restrict__ adj, float trans_weight,
                                                                         float rot_weight, float* __restrict__ v_adj, float* __restrict__ loss) {
    __shared__ double part[kCamRegThreads / 32];
    pdl_enter();
    const double wt = (double)trans_weight / num_cameras, wr = (double)rot_weight / num_cameras;
    double acc = 0.0;
    for (int j = threadIdx.x; j < num_cameras; j += kCamRegThreads) {
        const float* a = adj + (int64_t)j * 6;
        float* v = v_adj + (int64_t)j * 6;
        for (int h = 0; h < 2; ++h) {
            const double x = a[3 * h], y = a[3 * h + 1], z = a[3 * h + 2];
            const double n = sqrt(x * x + y * y + z * z), w = h ? wr : wt;
            acc += w * n;
            if (n > 0.0) {
                v[3 * h] += (float)(w * x / n);
                v[3 * h + 1] += (float)(w * y / n);
                v[3 * h + 2] += (float)(w * z / n);
            }
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = part[0];
        for (int w = 1; w < kCamRegThreads / 32; ++w) s += part[w];
        *loss = (float)s;
    }
}

}  // namespace qed

using namespace qed;

extern "C" int qed_viewmat_from_c2w(int C, int rows, const float* camera_to_worlds, float* viewmats, qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (C < 0 || !(rows == 3 || rows == 4)) return QED_ERR_BAD_ARG;
    if (C == 0) return QED_OK;
    if (!camera_to_worlds || !viewmats) return QED_ERR_BAD_ARG;
    viewmat_from_c2w_kernel<<<(C + 127) / 128, 128, 0, stream>>>(C, rows, camera_to_worlds, viewmats);
    QED_LAUNCH_CHECK();
    return QED_OK;
}

extern "C" int qed_viewmat_from_c2w_bwd(int C, int rows, const float* camera_to_worlds, const float* v_viewmats, float* v_camera_to_worlds,
                                        qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (C < 0 || !(rows == 3 || rows == 4)) return QED_ERR_BAD_ARG;
    if (C == 0) return QED_OK;
    if (!camera_to_worlds || !v_viewmats || !v_camera_to_worlds) return QED_ERR_BAD_ARG;
    QED_CUDA_TRY(launch_pdl(viewmat_from_c2w_bwd_kernel, dim3((C + 127) / 128), dim3(128), 0, stream, C, rows, camera_to_worlds, v_viewmats,
                            v_camera_to_worlds));
    return QED_OK;
}

extern "C" int qed_camera_opt_apply(int C, int rows, int num_cameras, const int32_t* camera_ids, const float* camera_to_worlds,
                                    const float* pose_adjustment, float* viewmats, qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (C < 0 || num_cameras < 1 || !(rows == 3 || rows == 4)) return QED_ERR_BAD_ARG;
    if (C == 0) return QED_OK;
    if (!camera_ids || !camera_to_worlds || !pose_adjustment || !viewmats) return QED_ERR_BAD_ARG;
    QED_CUDA_TRY(launch_pdl(camera_opt_apply_kernel, dim3((C + 127) / 128), dim3(128), 0, stream, C, rows, num_cameras, camera_ids,
                            camera_to_worlds, pose_adjustment, viewmats));
    return QED_OK;
}

extern "C" int qed_camera_opt_bwd(int C, int rows, int num_cameras, const int32_t* camera_ids, const float* camera_to_worlds,
                                  const float* pose_adjustment, const float* v_viewmats, float* v_pose_adjustment, qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (C < 0 || num_cameras < 1 || !(rows == 3 || rows == 4)) return QED_ERR_BAD_ARG;
    if (!pose_adjustment || !v_pose_adjustment || (C > 0 && (!camera_ids || !camera_to_worlds || !v_viewmats))) return QED_ERR_BAD_ARG;
    QED_CUDA_TRY(launch_pdl(camera_opt_bwd_kernel, dim3((num_cameras + 127) / 128), dim3(128), 0, stream, C, rows, num_cameras, camera_ids,
                            camera_to_worlds, pose_adjustment, v_viewmats, v_pose_adjustment));
    return QED_OK;
}

extern "C" int qed_camera_opt_reg(int num_cameras, const float* pose_adjustment, float trans_weight, float rot_weight, float* v_pose_adjustment,
                                  float* reg_loss, qed_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (num_cameras < 1 || !pose_adjustment || !v_pose_adjustment || !reg_loss) return QED_ERR_BAD_ARG;
    QED_CUDA_TRY(launch_pdl(camera_opt_reg_kernel, dim3(1), dim3(kCamRegThreads), 0, stream, num_cameras, pose_adjustment, trans_weight, rot_weight,
                            v_pose_adjustment, reg_loss));
    return QED_OK;
}
