// Trainable encoder-head / MLP element kernels (fp32): SpatialLearnedEmbeddings, Dropout,
// LayerNorm+tanh (forward and backward), column reductions for bias / scale gradients.
//
// Reference (relative to serl_launcher/serl_launcher):
//   vision/resnet_v1.py:81-116   SpatialLearnedEmbeddings: out[b, c*F+f] = sum_{h,w} feat[b,h,w,c] K[h,w,c,f]
//   vision/resnet_v1.py:352      nn.Dropout(0.1): where(mask, x / keep, 0)
//   vision/resnet_v1.py:371-374, common/encoding.py:65-70, networks/mlp.py:26-31
//                                Dense -> LayerNorm(eps 1e-6, var = E[x^2]-E[x]^2) -> tanh
// Restated in oracle/drq.py (encode, mlp2, layer_norm).
#include "common.cuh"
#include "serl_b200.h"

namespace serl {

// ---- SpatialLearnedEmbeddings forward: thread per (n, c), F == 8 --------------------------------
__global__ void sle_fwd_kernel(const float* __restrict__ feat, const float* __restrict__ kern,
                               const uint8_t* __restrict__ keep_mask, float keep, float* __restrict__ out,
                               int N, int P, int C, int ld_out) {
  pdl_prologue();
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N * C) return;
  const int n = e / C, c = e - n * C;
  float acc[8];
#pragma unroll
  for (int f = 0; f < 8; ++f) acc[f] = 0.f;
  for (int p = 0; p < P; ++p) {
    const float v = feat[((size_t)n * P + p) * C + c];
    const float4 k0 = *reinterpret_cast<const float4*>(kern + ((size_t)p * C + c) * 8);
    const float4 k1 = *reinterpret_cast<const float4*>(kern + ((size_t)p * C + c) * 8 + 4);
    acc[0] = fmaf(v, k0.x, acc[0]); acc[1] = fmaf(v, k0.y, acc[1]); acc[2] = fmaf(v, k0.z, acc[2]); acc[3] = fmaf(v, k0.w, acc[3]);
    acc[4] = fmaf(v, k1.x, acc[4]); acc[5] = fmaf(v, k1.y, acc[5]); acc[6] = fmaf(v, k1.z, acc[6]); acc[7] = fmaf(v, k1.w, acc[7]);
  }
  if (keep_mask) {
    const uint8_t* mk = keep_mask + (size_t)n * C * 8 + c * 8;
#pragma unroll
    for (int f = 0; f < 8; ++f) acc[f] = mk[f] ? acc[f] / keep : 0.f;
  }
  float* o = out + (size_t)n * ld_out + c * 8;
  *reinterpret_cast<float4*>(o) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  *reinterpret_cast<float4*>(o + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
}

// ---- SLE kernel gradient: partial[chunk][p][c][f] = sum_{n in chunk} feat[n,p,c] * dout[n, c*8+f] ----
__global__ void sle_bwd_partial_kernel(const float* __restrict__ feat, const float* __restrict__ dout,
                                       float* __restrict__ partial, int N, int P, int C, int ld_dout, int chunks) {
  pdl_prologue();
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P * C) return;
  const int p = e / C, c = e - p * C;
  const int ch = blockIdx.y;
  const int per = ceil_div(N, chunks);
  const int n0 = ch * per, n1 = min(N, n0 + per);
  float acc[8];
#pragma unroll
  for (int f = 0; f < 8; ++f) acc[f] = 0.f;
  for (int n = n0; n < n1; ++n) {
    const float v = feat[((size_t)n * P + p) * C + c];
    const float4 d0 = *reinterpret_cast<const float4*>(dout + (size_t)n * ld_dout + c * 8);
    const float4 d1 = *reinterpret_cast<const float4*>(dout + (size_t)n * ld_dout + c * 8 + 4);
    acc[0] = fmaf(v, d0.x, acc[0]); acc[1] = fmaf(v, d0.y, acc[1]); acc[2] = fmaf(v, d0.z, acc[2]); acc[3] = fmaf(v, d0.w, acc[3]);
    acc[4] = fmaf(v, d1.x, acc[4]); acc[5] = fmaf(v, d1.y, acc[5]); acc[6] = fmaf(v, d1.z, acc[6]); acc[7] = fmaf(v, d1.w, acc[7]);
  }
  float* o = partial + ((size_t)ch * P * C + e) * 8;
  *reinterpret_cast<float4*>(o) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  *reinterpret_cast<float4*>(o + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
}

// ---- out[g][d] = sum_{r < rows} x[(g*rows + r) * ld + d] --------------------------------------------------------
// block = 32 columns x 8 row-slices (coalesced 128-byte row reads), fixed-order tree over the slices: deterministic.
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ x, float* __restrict__ out, int groups, int rows, int D,
                                                     long long ld, int accumulate) {
  pdl_prologue();
  __shared__ float red[8][33];
  const int cx = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int cblocks = ceil_div(D, 32);
  const int g = blockIdx.x / cblocks, d = (blockIdx.x - g * cblocks) * 32 + cx;
  float s = 0.f;
  if (d < D) {
    const float* p = x + (size_t)g * rows * ld + d;
    for (int r = sl; r < rows; r += 8) s += p[(size_t)r * ld];
  }
  red[sl][cx] = s;
  __syncthreads();
  if (sl == 0 && d < D) {
    float t = red[0][cx];
#pragma unroll
    for (int k = 1; k < 8; ++k) t += red[k][cx];
    const size_t e = (size_t)g * D + d;
    out[e] = accumulate ? out[e] + t : t;
  }
}

// ---- LayerNorm + tanh forward: warp per row -------------------------------------------------------
// rows R = groups * rows_per_group; scale/bias of row r at (r / rows_per_group) * group_stride.
__global__ void ln_tanh_fwd_kernel(const float* __restrict__ z, int ld_z, const float* __restrict__ scale,
                                   const float* __restrict__ bias, int rows_per_group, int group_stride,
                                   float* __restrict__ out, int ld_out, float* __restrict__ xhat, float* __restrict__ rstd_out,
                                   int R, int D, float eps) {
  pdl_prologue();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= R) return;
  const float* zr = z + (size_t)row * ld_z;
  float s = 0.f, ss = 0.f;
  for (int d = lane; d < D; d += 32) { float v = zr[d]; s += v; ss += v * v; }
  s = warp_sum(s); ss = warp_sum(ss);
  const float mean = s / (float)D;
  const float var = fmaxf(ss / (float)D - mean * mean, 0.f);
  const float rstd = rsqrtf(var + eps);
  const int g = row / rows_per_group;
  const float* sc = scale + (size_t)g * group_stride;
  const float* bi = bias + (size_t)g * group_stride;
  for (int d = lane; d < D; d += 32) {
    const float xh = (zr[d] - mean) * rstd;
    out[(size_t)row * ld_out + d] = tanhf(xh * sc[d] + bi[d]);
    if (xhat) xhat[(size_t)row * D + d] = xh;
  }
  if (rstd_out && lane == 0) rstd_out[row] = rstd;
}

// ---- LayerNorm + tanh backward: warp per row ------------------------------------------------------
// dy = dt * (1 - t^2);  dz = rstd * (dy*scale - mean(dy*scale) - xhat * mean(dy*scale*xhat));  dy kept for param grads.
__global__ void ln_tanh_bwd_kernel(const float* __restrict__ dt, int ld_dt, const float* __restrict__ t, int ld_t,
                                   const float* __restrict__ xhat, const float* __restrict__ rstd,
                                   const float* __restrict__ scale, int rows_per_group, int group_stride,
                                   float* __restrict__ dz, float* __restrict__ dy_out, int R, int D) {
  pdl_prologue();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= R) return;
  const float* sc = scale + (size_t)(row / rows_per_group) * group_stride;
  float m1 = 0.f, m2 = 0.f;
  for (int d = lane; d < D; d += 32) {
    const float tv = t[(size_t)row * ld_t + d];
    const float dy = dt[(size_t)row * ld_dt + d] * (1.f - tv * tv);
    const float dxh = dy * sc[d];
    m1 += dxh; m2 += dxh * xhat[(size_t)row * D + d];
    dy_out[(size_t)row * D + d] = dy;
  }
  m1 = warp_sum(m1) / (float)D; m2 = warp_sum(m2) / (float)D;
  const float rs = rstd[row];
  for (int d = lane; d < D; d += 32) {
    const float dxh = dy_out[(size_t)row * D + d] * sc[d];
    dz[(size_t)row * D + d] = rs * (dxh - m1 - xhat[(size_t)row * D + d] * m2);
  }
}

// ---- dscale[g][d] = sum_r dy*xhat ; dbias[g][d] = sum_r dy   (same 32 x 8 block shape as colsum) -----------------
__global__ void __launch_bounds__(256) ln_param_grad_kernel(const float* __restrict__ dy, const float* __restrict__ xhat,
                                                            float* __restrict__ dscale, float* __restrict__ dbias, int groups, int rows, int D) {
  pdl_prologue();
  __shared__ float ra[8][33], rb[8][33];
  const int cx = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int cblocks = ceil_div(D, 32);
  const int g = blockIdx.x / cblocks, d = (blockIdx.x - g * cblocks) * 32 + cx;
  float a = 0.f, b = 0.f;
  if (d < D) {
    for (int r = sl; r < rows; r += 8) {
      const size_t off = ((size_t)g * rows + r) * D + d;
      const float v = dy[off];
      a += v * xhat[off]; b += v;
    }
  }
  ra[sl][cx] = a; rb[sl][cx] = b;
  __syncthreads();
  if (sl == 0 && d < D) {
    float ta = ra[0][cx], tb = rb[0][cx];
#pragma unroll
    for (int k = 1; k < 8; ++k) { ta += ra[k][cx]; tb += rb[k][cx]; }
    dscale[(size_t)g * D + d] = ta; dbias[(size_t)g * D + d] = tb;
  }
}

// ---- reward classifier hidden layer: Dense -> Dropout -> LayerNorm -> ReLU (networks/reward_classifier.py:22-26) ----------
// Forward, warp per row: d = keep_mask ? z / keep : 0, LayerNorm statistics of d (fast variance), out = relu(xhat*scale + bias).
__global__ void ln_relu_fwd_kernel(const float* __restrict__ z, int ld_z, const uint8_t* __restrict__ keep_mask, float keep,
                                   const float* __restrict__ scale, const float* __restrict__ bias, float* __restrict__ out, int ld_out,
                                   float* __restrict__ xhat, float* __restrict__ rstd_out, int R, int D, float eps) {
  pdl_prologue();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= R) return;
  float v[8];
  float s = 0.f, ss = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int d = lane + 32 * j;
    v[j] = 0.f;
    if (d < D) {
      float x = z[(size_t)row * ld_z + d];
      if (keep_mask) x = keep_mask[(size_t)row * D + d] ? x / keep : 0.f;
      v[j] = x; s += x; ss += x * x;
    }
  }
  s = warp_sum(s); ss = warp_sum(ss);
  const float mean = s / (float)D;
  const float var = fmaxf(ss / (float)D - mean * mean, 0.f);
  const float rstd = rsqrtf(var + eps);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int d = lane + 32 * j;
    if (d < D) {
      const float xh = (v[j] - mean) * rstd;
      out[(size_t)row * ld_out + d] = fmaxf(fmaf(xh, scale[d], bias[d]), 0.f);
      if (xhat) xhat[(size_t)row * D + d] = xh;
    }
  }
  if (rstd_out && lane == 0) rstd_out[row] = rstd;
}

// Backward, warp per row (serves the fp32 chain and the LN_RELU_HEAD epilogue of tgemm.cu, which saves the same xhat / rstd):
// dt = upstream or dlogit * w;  dy = dt * [xhat*scale + bias > 0];  dd = rstd * (dy*scale - mean(dy*scale) - xhat * mean(dy*scale*xhat));
// dz = keep_mask ? dd / keep : 0.
__global__ void __launch_bounds__(256) ln_relu_bwd_kernel(const float* __restrict__ dt, int ld_dt, const float* __restrict__ dlogit,
                                                          const float* __restrict__ head_w, const float* __restrict__ xhat,
                                                          const float* __restrict__ rstd, const float* __restrict__ scale,
                                                          const float* __restrict__ bias, const uint8_t* __restrict__ keep_mask, float keep,
                                                          float* __restrict__ dz, float* __restrict__ dy_out, int R, int D) {
  pdl_prologue();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= R) return;
  const float dl = dt ? 0.f : dlogit[row];
  float dy[8], xh[8];
  float m1 = 0.f, m2 = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int d = lane + 32 * j;
    dy[j] = 0.f; xh[j] = 0.f;
    if (d < D) {
      xh[j] = xhat[(size_t)row * D + d];
      const float g = dt ? dt[(size_t)row * ld_dt + d] : dl * head_w[d];
      dy[j] = fmaf(xh[j], scale[d], bias[d]) > 0.f ? g : 0.f;
      const float dxh = dy[j] * scale[d];
      m1 += dxh; m2 += dxh * xh[j];
      if (dy_out) dy_out[(size_t)row * D + d] = dy[j];
    }
  }
  m1 = warp_sum(m1) / (float)D; m2 = warp_sum(m2) / (float)D;
  const float rs = rstd[row];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int d = lane + 32 * j;
    if (d < D) {
      float g = rs * (dy[j] * scale[d] - m1 - xh[j] * m2);
      if (keep_mask) g = keep_mask[(size_t)row * D + d] ? g / keep : 0.f;
      dz[(size_t)row * D + d] = g;
    }
  }
}

// ---- Dropout backward in place: x = mask ? x / keep : 0 (the SLE output's gradient of a train=True pass before the kernel gradient) --
__global__ void dropout_bwd_kernel(float* __restrict__ x, const uint8_t* __restrict__ mask, float keep, long long n) {
  pdl_prologue();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    x[i] = mask[i] ? x[i] / keep : 0.f;
}

// ---- strided 2-D copy (concat helper) -------------------------------------------------------------
__global__ void copy2d_kernel(const float* __restrict__ src, long long ld_src, float* __restrict__ dst, long long ld_dst, int R, int D) {
  pdl_prologue();
  const size_t total = (size_t)R * D;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(e / D), d = (int)(e - (size_t)r * D);
    dst[(size_t)r * ld_dst + d] = src[(size_t)r * ld_src + d];
  }
}

}  // namespace serl

using namespace serl;
#define ST(s) static_cast<cudaStream_t>(s)

extern "C" int serl_sle_fwd(const float* feat, const float* kernel, const uint8_t* keep_mask, float keep, float* out,
                            int N, int P, int C, int F, int ld_out, void* stream) {
  if (F != 8 || (ld_out & 3)) { set_last_error("serl_sle_fwd: num_features must be 8 and ld_out %% 4 == 0"); return SERL_ERR_UNSUPPORTED; }
  launch_k(sle_fwd_kernel, ceil_div(N * C, 128), 128, 0, ST(stream), feat, kernel, keep_mask, keep, out, N, P, C, ld_out);
  return check_launch("sle_fwd_kernel");
}

extern "C" int serl_sle_bwd_kernel_grad(const float* feat, const float* dout, float* dkernel, float* workspace,
                                        size_t workspace_bytes, int N, int P, int C, int F, int ld_dout, void* stream) {
  if (F != 8 || (ld_dout & 3)) { set_last_error("serl_sle_bwd_kernel_grad: num_features must be 8"); return SERL_ERR_UNSUPPORTED; }
  int chunks = N >= 64 ? 16 : 1;
  const size_t per = (size_t)P * C * F * sizeof(float);
  while (chunks > 1 && per * chunks > workspace_bytes) chunks >>= 1;
  if (!workspace || per * chunks > workspace_bytes) { set_last_error("serl_sle_bwd_kernel_grad: workspace too small (%zu needed)", per); return SERL_ERR_INVALID; }
  dim3 grid(ceil_div(P * C, 128), chunks);
  launch_k(sle_bwd_partial_kernel, grid, 128, 0, ST(stream), feat, dout, workspace, N, P, C, ld_dout, chunks);
  if (int e = check_launch("sle_bwd_partial_kernel")) return e;
  const int D = P * C * F;
  launch_k(colsum_kernel, ceil_div(D, 32), 256, 0, ST(stream), workspace, dkernel, 1, chunks, D, D, 0);
  return check_launch("colsum_kernel(sle)");
}

extern "C" int serl_colsum_f32(const float* x, float* out, int groups, int rows, int D, long long ld, int accumulate, void* stream) {
  launch_k(colsum_kernel, groups * ceil_div(D, 32), 256, 0, ST(stream), x, out, groups, rows, D, ld, accumulate);
  return check_launch("colsum_kernel");
}

extern "C" int serl_layernorm_tanh_fwd(const float* z, int ld_z, const float* scale, const float* bias, int rows_per_group,
                                       int group_stride, float* out, int ld_out, float* xhat, float* rstd, int R, int D,
                                       float eps, void* stream) {
  launch_k(ln_tanh_fwd_kernel, ceil_div(R, 8), 256, 0, ST(stream), z, ld_z, scale, bias, rows_per_group, group_stride, out, ld_out,
                                                             xhat, rstd, R, D, eps);
  return check_launch("ln_tanh_fwd_kernel");
}

extern "C" int serl_layernorm_tanh_bwd(const float* dt, int ld_dt, const float* t, int ld_t, const float* xhat, const float* rstd,
                                       const float* scale, int rows_per_group, int group_stride, float* dz, float* dy,
                                       float* dscale, float* dbias, int R, int D, void* stream) {
  launch_k(ln_tanh_bwd_kernel, ceil_div(R, 8), 256, 0, ST(stream), dt, ld_dt, t, ld_t, xhat, rstd, scale, rows_per_group, group_stride,
                                                             dz, dy, R, D);
  if (int e = check_launch("ln_tanh_bwd_kernel")) return e;
  if (dscale && dbias) {
    const int groups = R / rows_per_group;
    launch_k(ln_param_grad_kernel, groups * ceil_div(D, 32), 256, 0, ST(stream), dy, xhat, dscale, dbias, groups, rows_per_group, D);
    return check_launch("ln_param_grad_kernel");
  }
  return SERL_OK;
}

// the parameter-gradient half of serl_layernorm_tanh_bwd on its own (dy, xhat as that call left them): lets the caller put it
// on a side stream, off the dz -> next-layer chain
extern "C" int serl_layernorm_param_grad(const float* dy, const float* xhat, float* dscale, float* dbias, int rows_per_group, int R, int D,
                                         void* stream) {
  if (!dy || !xhat || !dscale || !dbias || rows_per_group < 1 || R % rows_per_group != 0) {
    set_last_error("serl_layernorm_param_grad: invalid arguments"); return SERL_ERR_INVALID;
  }
  const int groups = R / rows_per_group;
  launch_k(ln_param_grad_kernel, groups * ceil_div(D, 32), 256, 0, ST(stream), dy, xhat, dscale, dbias, groups, rows_per_group, D);
  return check_launch("ln_param_grad_kernel");
}

extern "C" int serl_copy2d_f32(const float* src, long long ld_src, float* dst, long long ld_dst, int R, int D, void* stream) {
  size_t total = (size_t)R * D;
  int blocks = (int)((total + 255) / 256); if (blocks > 1184) blocks = 1184; if (blocks < 1) blocks = 1;
  launch_k(copy2d_kernel, blocks, 256, 0, ST(stream), src, ld_src, dst, ld_dst, R, D);
  return check_launch("copy2d_kernel");
}

extern "C" int serl_layernorm_relu_fwd(const float* z, int ld_z, const uint8_t* keep_mask, float keep, const float* scale, const float* bias,
                                       float* out, int ld_out, float* xhat, float* rstd, int R, int D, float eps, void* stream) {
  if (!z || !scale || !bias || !out || R < 1 || D < 1 || D > 256 || (keep_mask && !(keep > 0.f))) {
    set_last_error("serl_layernorm_relu_fwd: invalid arguments (D <= 256, keep > 0 with a mask)"); return SERL_ERR_INVALID;
  }
  launch_k(ln_relu_fwd_kernel, ceil_div(R, 8), 256, 0, ST(stream), z, ld_z, keep_mask, keep, scale, bias, out, ld_out, xhat, rstd, R, D, eps);
  return check_launch("ln_relu_fwd_kernel");
}

extern "C" int serl_layernorm_relu_bwd(const float* dt, int ld_dt, const float* dlogit, const float* head_w, const float* xhat, const float* rstd,
                                       const float* scale, const float* bias, const uint8_t* keep_mask, float keep, float* dz, float* dy,
                                       int R, int D, void* stream) {
  if ((!dt && (!dlogit || !head_w)) || !xhat || !rstd || !scale || !bias || !dz || R < 1 || D < 1 || D > 256 || (keep_mask && !(keep > 0.f))) {
    set_last_error("serl_layernorm_relu_bwd: invalid arguments (dt, or dlogit + head_w; D <= 256)"); return SERL_ERR_INVALID;
  }
  launch_k(ln_relu_bwd_kernel, ceil_div(R, 8), 256, 0, ST(stream), dt, ld_dt, dlogit, head_w, xhat, rstd, scale, bias, keep_mask, keep, dz, dy, R, D);
  return check_launch("ln_relu_bwd_kernel");
}

extern "C" int serl_dropout_bwd(float* x, const uint8_t* keep_mask, float keep, long long n, void* stream) {
  if (!x || !keep_mask || n < 1 || !(keep > 0.f)) { set_last_error("serl_dropout_bwd: invalid arguments"); return SERL_ERR_INVALID; }
  long long blocks = (n + 255) / 256; if (blocks > 2368) blocks = 2368;
  launch_k(dropout_bwd_kernel, (int)blocks, 256, 0, ST(stream), x, keep_mask, keep, n);
  return check_launch("dropout_bwd_kernel");
}
