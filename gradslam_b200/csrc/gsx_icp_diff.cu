// Differentiable small ops of the ICP / gradICP loop for sm_100a (K7 forward + backward, and the rigid transform of
// the source cloud).  They replace the ~80 tiny ATen kernels per iteration that PyTorch's tape records for
//   solve_linear_system      gradslam/odometry/icputils.py:22-90
//   se3_exp                  gradslam/geometry/se3utils.py:77-115
//   LM accept / reject       gradslam/odometry/icputils.py:356-365
//   gradLM gates             gradslam/odometry/icputils.py:519-543
//   transform_pointcloud     gradslam/geometry/geometryutils.py:737-794
// The forward arithmetic is the one of the fused loop (k_icp_solve / k_icp_update in gsx_icp.cu), written once as
// templates over the scalar type.  The backward kernels evaluate the same templates on dual numbers: lane j seeds input
// j, so it obtains column j of the Jacobian and one dot product with the upstream gradient gives d(loss)/d(input j).
// The functions have 25-29 inputs and a few hundred operations: one warp-sized launch, no reductions, no atomics.
#include "gsx_common.cuh"
#include "gsx_icp_diff.cuh"
#include "../../include/gsx.h"

namespace gsx {

__global__ void k_solve_fwd(const float *sums, const float *damp, float *xi, float *dT, int n) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  float in[kSolveIn], out[kSolveOut];
  for (int i = 0; i < 28; ++i) in[i] = sums[e * 28 + i];
  in[28] = damp[e];
  solve_step_t<float>(in, out);
  for (int i = 0; i < 6; ++i) xi[e * 6 + i] = out[i];
  for (int i = 0; i < 16; ++i) dT[e * 16 + i] = out[6 + i];
}

// one warp per element, lane j -> d(loss)/d(input j)
__global__ void __launch_bounds__(32) k_solve_bwd(const float *sums, const float *damp, const float *g_xi,
                                                  const float *g_dT, float *g_sums, float *g_damp) {
  const int e = blockIdx.x, j = threadIdx.x;
  if (j >= kSolveIn) return;
  Dual in[kSolveIn], out[kSolveOut];
  for (int i = 0; i < 28; ++i) in[i] = mk(sums[e * 28 + i], i == j ? 1.0f : 0.0f);
  in[28] = mk(damp[e], j == 28 ? 1.0f : 0.0f);
  solve_step_t<Dual>(in, out);
  float g = 0.0f;
  if (g_xi)
    for (int i = 0; i < 6; ++i) g += g_xi[e * 6 + i] * out[i].d;
  if (g_dT)
    for (int i = 0; i < 16; ++i) g += g_dT[e * 16 + i] * out[6 + i].d;
  if (j < 28) g_sums[e * 28 + j] = g;
  else g_damp[e] = g;
}

__device__ __forceinline__ void load_update_inputs(const float *xi, const float *err, const float *new_err,
                                                   const float *damp, const float *T, int e, float *in) {
  for (int i = 0; i < 6; ++i) in[i] = xi[e * 6 + i];
  in[6] = err[e];
  in[7] = new_err[e];
  in[8] = damp[e];
  for (int i = 0; i < 16; ++i) in[9 + i] = T[e * 16 + i];
}

__global__ void k_update_fwd(const float *xi, const float *err, const float *new_err, const float *damp, const float *T,
                             UpdateParams u, float *damp_out, float *dT_out, float *T_out, int n) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  float in[kUpdateIn], out[kUpdateOut];
  load_update_inputs(xi, err, new_err, damp, T, e, in);
  update_step_t<float>(in, out, u);
  damp_out[e] = out[0];
  for (int i = 0; i < 16; ++i) {
    dT_out[e * 16 + i] = out[1 + i];
    T_out[e * 16 + i] = out[17 + i];
  }
}

__global__ void __launch_bounds__(32) k_update_bwd(const float *xi, const float *err, const float *new_err,
                                                   const float *damp, const float *T, UpdateParams u,
                                                   const float *g_damp_out, const float *g_dT_out, const float *g_T_out,
                                                   float *g_xi, float *g_err, float *g_new_err, float *g_damp,
                                                   float *g_T) {
  const int e = blockIdx.x, j = threadIdx.x;
  if (j >= kUpdateIn) return;
  float inf[kUpdateIn];
  load_update_inputs(xi, err, new_err, damp, T, e, inf);
  Dual in[kUpdateIn], out[kUpdateOut];
  for (int i = 0; i < kUpdateIn; ++i) in[i] = mk(inf[i], i == j ? 1.0f : 0.0f);
  update_step_t<Dual>(in, out, u);
  float g = 0.0f;
  if (g_damp_out) g += g_damp_out[e] * out[0].d;
  if (g_dT_out)
    for (int i = 0; i < 16; ++i) g += g_dT_out[e * 16 + i] * out[1 + i].d;
  if (g_T_out)
    for (int i = 0; i < 16; ++i) g += g_T_out[e * 16 + i] * out[17 + i].d;
  if (j < 6) g_xi[e * 6 + j] = g;
  else if (j == 6) g_err[e] = g;
  else if (j == 7) g_new_err[e] = g;
  else if (j == 8) g_damp[e] = g;
  else g_T[e * 16 + (j - 9)] = g;
}

// ---- rigid transform of a cloud: out = R p + t (geometryutils.py:737-794), canonical left-to-right sums ------------
constexpr int kRtBlock = 256;
// (batched: element b = blockIdx.y owns `stride` rows and T + 16 b; counts may be null = `stride` rows each.  Padding rows
//  of a batched call are written as zeros, so the padded cloud stays a valid zero-padded tensor.)
__global__ void __launch_bounds__(kRtBlock) k_rigid_fwd(const float *src, int64_t stride, const int32_t *counts,
                                                        const float *T, float *out) {
  __shared__ Rigid s_T;
  const int b = blockIdx.y;
  const int64_t n = counts ? counts[b] : stride;
  src += (int64_t)b * stride * 3;
  out += (int64_t)b * stride * 3;
  if (threadIdx.x == 0) s_T = load_rigid(T + b * 16);
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * kRtBlock + threadIdx.x;
  if (i >= stride) return;
  if (i >= n) {
    out[i * 3] = out[i * 3 + 1] = out[i * 3 + 2] = 0.0f;
    return;
  }
  const float3 q = rigid_apply(s_T, src[i * 3], src[i * 3 + 1], src[i * 3 + 2]);
  out[i * 3] = q.x;
  out[i * 3 + 1] = q.y;
  out[i * 3 + 2] = q.z;
}

// g_src = R^T g; per-block partial sums of g (x) [p; 1] (12 numbers) in a fixed order, reduced by k_rigid_bwd_reduce
__global__ void __launch_bounds__(kRtBlock) k_rigid_bwd(const float *src, int64_t stride, const int32_t *counts,
                                                        const float *T, const float *g_out, float *g_src,
                                                        float *partials) {
  __shared__ Rigid s_T;
  __shared__ float s_red[kRtBlock / 32][12];
  const int b = blockIdx.y;
  const int64_t n = counts ? counts[b] : stride;
  src += (int64_t)b * stride * 3;
  g_out += (int64_t)b * stride * 3;
  g_src += (int64_t)b * stride * 3;
  partials += (int64_t)b * gridDim.x * 12;
  if (threadIdx.x == 0) s_T = load_rigid(T + b * 16);
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * kRtBlock + threadIdx.x;
  if (i >= n && i < stride) g_src[i * 3] = g_src[i * 3 + 1] = g_src[i * 3 + 2] = 0.0f;
  float acc[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) acc[k] = 0.0f;
  if (i < n) {
    const float gx = g_out[i * 3], gy = g_out[i * 3 + 1], gz = g_out[i * 3 + 2];
    const float px = src[i * 3], py = src[i * 3 + 1], pz = src[i * 3 + 2];
    g_src[i * 3] = dot3(s_T.r[0], s_T.r[3], s_T.r[6], gx, gy, gz);
    g_src[i * 3 + 1] = dot3(s_T.r[1], s_T.r[4], s_T.r[7], gx, gy, gz);
    g_src[i * 3 + 2] = dot3(s_T.r[2], s_T.r[5], s_T.r[8], gx, gy, gz);
    const float g[3] = {gx, gy, gz};
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      acc[r * 4 + 0] = g[r] * px;
      acc[r * 4 + 1] = g[r] * py;
      acc[r * 4 + 2] = g[r] * pz;
      acc[r * 4 + 3] = g[r];
    }
  }
#pragma unroll
  for (int k = 0; k < 12; ++k) {
    float v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    acc[k] = v;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 12; ++k) s_red[warp][k] = acc[k];
  }
  __syncthreads();
  if (threadIdx.x < 12) {
    float v = 0.0f;
#pragma unroll
    for (int w = 0; w < kRtBlock / 32; ++w) v += s_red[w][threadIdx.x];
    partials[(int64_t)blockIdx.x * 12 + threadIdx.x] = v;
  }
}

__global__ void k_rigid_bwd_reduce(const float *partials, int nblocks, float *g_T) {
  partials += (int64_t)blockIdx.x * nblocks * 12;  // (one block per batch element)
  g_T += (int64_t)blockIdx.x * 16;
  const int k = threadIdx.x;
  if (k < 12) {
    float v = 0.0f;
    for (int j = 0; j < nblocks; ++j) v += partials[(int64_t)j * 12 + k];
    g_T[k] = v;
  } else if (k < 16) {
    g_T[k] = 0.0f;  // the bottom row of T does not enter the transform
  }
}

}  // namespace gsx

using namespace gsx;

extern "C" int gsx_icp_solve_fwd(const float *sums, const float *damp, int n, float *xi_out, float *dT_out,
                                 void *stream) {
  GSX_CHECK_ARG(n >= 0, "gsx_icp_solve_fwd: negative count");
  if (n == 0) return 0;
  GSX_CHECK_ARG(sums && damp && xi_out && dT_out, "gsx_icp_solve_fwd: null pointer");
  k_solve_fwd<<<(n + 31) / 32, 32, 0, (cudaStream_t)stream>>>(sums, damp, xi_out, dT_out, n);
  GSX_CHECK_LAUNCH("gsx_icp_solve_fwd");
  return 0;
}

extern "C" int gsx_icp_solve_bwd(const float *sums, const float *damp, int n, const float *g_xi, const float *g_dT,
                                 float *g_sums, float *g_damp, void *stream) {
  GSX_CHECK_ARG(n >= 0, "gsx_icp_solve_bwd: negative count");
  if (n == 0) return 0;
  GSX_CHECK_ARG(sums && damp && g_sums && g_damp, "gsx_icp_solve_bwd: null pointer");
  k_solve_bwd<<<n, 32, 0, (cudaStream_t)stream>>>(sums, damp, g_xi, g_dT, g_sums, g_damp);
  GSX_CHECK_LAUNCH("gsx_icp_solve_bwd");
  return 0;
}

static bool make_update_params(int mode, float lambda_max, float Bp, float B2p, float nu, UpdateParams *u) {
  if ((mode != 0 && mode != 1) || !(lambda_max > 0.0f) || nu == 0.0f) return false;
  *u = UpdateParams{mode, 1.0f / lambda_max, lambda_max, Bp, B2p, 1.0f / nu};
  return true;
}

extern "C" int gsx_icp_update_fwd(const float *xi, const float *err, const float *new_err, const float *damp,
                                  const float *T, int n, int mode, float lambda_max, float Bp, float B2p, float nu,
                                  float *damp_out, float *dT_out, float *T_out, void *stream) {
  GSX_CHECK_ARG(n >= 0, "gsx_icp_update_fwd: negative count");
  if (n == 0) return 0;
  GSX_CHECK_ARG(xi && err && new_err && damp && T && damp_out && dT_out && T_out, "gsx_icp_update_fwd: null pointer");
  UpdateParams u;
  GSX_CHECK_ARG(make_update_params(mode, lambda_max, Bp, B2p, nu, &u), "gsx_icp_update_fwd: bad mode / gate parameters");
  k_update_fwd<<<(n + 31) / 32, 32, 0, (cudaStream_t)stream>>>(xi, err, new_err, damp, T, u, damp_out, dT_out, T_out, n);
  GSX_CHECK_LAUNCH("gsx_icp_update_fwd");
  return 0;
}

extern "C" int gsx_icp_update_bwd(const float *xi, const float *err, const float *new_err, const float *damp,
                                  const float *T, int n, int mode, float lambda_max, float Bp, float B2p, float nu,
                                  const float *g_damp_out, const float *g_dT_out, const float *g_T_out, float *g_xi,
                                  float *g_err, float *g_new_err, float *g_damp, float *g_T, void *stream) {
  GSX_CHECK_ARG(n >= 0, "gsx_icp_update_bwd: negative count");
  if (n == 0) return 0;
  GSX_CHECK_ARG(xi && err && new_err && damp && T && g_xi && g_err && g_new_err && g_damp && g_T,
                "gsx_icp_update_bwd: null pointer");
  UpdateParams u;
  GSX_CHECK_ARG(make_update_params(mode, lambda_max, Bp, B2p, nu, &u), "gsx_icp_update_bwd: bad mode / gate parameters");
  k_update_bwd<<<n, 32, 0, (cudaStream_t)stream>>>(xi, err, new_err, damp, T, u, g_damp_out, g_dT_out, g_T_out, g_xi,
                                                   g_err, g_new_err, g_damp, g_T);
  GSX_CHECK_LAUNCH("gsx_icp_update_bwd");
  return 0;
}

extern "C" int gsx_rigid_transform_batched_fwd(const float *points, const int32_t *counts, int64_t stride, int B,
                                               const float *T, float *out, void *stream) {
  GSX_CHECK_ARG(B >= 1 && stride >= 1, "gsx_rigid_transform_batched_fwd: bad sizes");
  GSX_CHECK_ARG(points && T && out, "gsx_rigid_transform_batched_fwd: null pointer");
  k_rigid_fwd<<<dim3((unsigned)((stride + kRtBlock - 1) / kRtBlock), (unsigned)B), kRtBlock, 0, (cudaStream_t)stream>>>(
      points, stride, counts, T, out);
  GSX_CHECK_LAUNCH("gsx_rigid_transform_batched_fwd");
  return 0;
}

extern "C" int gsx_rigid_transform_batched_bwd(const float *points, const int32_t *counts, int64_t stride, int B,
                                               const float *T, const float *g_out, float *g_points, float *g_T,
                                               void *scratch, int64_t scratch_bytes, void *stream) {
  GSX_CHECK_ARG(B >= 1 && stride >= 1, "gsx_rigid_transform_batched_bwd: bad sizes");
  GSX_CHECK_ARG(points && T && g_out && g_points && g_T && scratch, "gsx_rigid_transform_batched_bwd: null pointer");
  GSX_CHECK_ARG(scratch_bytes >= (int64_t)B * gsx_rigid_transform_bwd_scratch_bytes(stride),
                "gsx_rigid_transform_batched_bwd: scratch too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int nblk = (int)((stride + kRtBlock - 1) / kRtBlock);
  k_rigid_bwd<<<dim3((unsigned)nblk, (unsigned)B), kRtBlock, 0, st>>>(points, stride, counts, T, g_out, g_points,
                                                                      (float *)scratch);
  k_rigid_bwd_reduce<<<B, 32, 0, st>>>((const float *)scratch, nblk, g_T);
  GSX_CHECK_LAUNCH("gsx_rigid_transform_batched_bwd");
  return 0;
}

extern "C" int64_t gsx_rigid_transform_bwd_scratch_bytes(int64_t n) {
  if (n < 0) return -1;
  return ((n + kRtBlock - 1) / kRtBlock) * 12 * 4 + 256;
}
