// (a1) camera-to-world -> gsplat world-to-camera, the `get_viewmat` of qed_splatter/model.py:22-38:
//   R = c2w[:, :3, :3] * [1, -1, -1]   (flip the y and z COLUMNS: nerfstudio/OpenGL -> gsplat/OpenCV camera axes)
//   viewmat = [[R^T, -R^T T], [0 0 0 1]]          (analytic inverse of a rigid transform)
// One thread per camera; every product and sum is an individually rounded IEEE operation in a fixed order
// (((r0 t0 + r1 t1) + r2 t2), negated), which is what oracle/torch_impl.py::get_viewmat's float32 bmm evaluates to on
// the host cores, so the result is bit-identical to the oracle (tests/test_gpu_data_side.py).
#include "common.cuh"

namespace qed {

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
    float* v = viewmats + (int64_t)c * 16;
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
