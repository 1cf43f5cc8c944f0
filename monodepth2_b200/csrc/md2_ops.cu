// md2_ops.cu - per-layer sm_100a kernels behind the layers.py drop-in classes
// (include/md2_loss.h, "per-layer entry points").  These keep the reference's unfused
// call graph working (trainer.py calling BackprojectDepth -> Project3D -> grid_sample ->
// SSIM ...); the fused md2_view_synthesis_loss is the fast path.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>

#include "../../include/md2_loss.h"
#include "md2_core.cuh"

namespace {

constexpr int kT = 256;
inline int blocks_for(long long n) { return (int)((n + kT - 1) / kT); }
inline int rc(cudaError_t e) { return e == cudaSuccess ? MD2_OK : MD2_ERR_CUDA; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// block-wide sum; result valid in thread 0.  blockDim.x == kT.
__device__ __forceinline__ float block_sum(float v) {
  __shared__ float part[32];
  __syncthreads();
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    v = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.f;
    v = warp_sum(v);
  }
  return v;
}

// ---------------------------------------------------------------- disp_to_depth (layers.py:16-25)
__global__ void k_disp_to_depth(const float* __restrict__ disp, float a, float c, float* scaled,
                                float* depth, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float sd = __fadd_rn(a, __fmul_rn(c, disp[i]));
  if (scaled) scaled[i] = sd;
  if (depth) depth[i] = __frcp_rn(sd);
}
__global__ void k_disp_to_depth_bwd(const float* __restrict__ disp, float a, float c,
                                    const float* gs, const float* gd, float* gdisp, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float sd = __fadd_rn(a, __fmul_rn(c, disp[i]));
  float g = 0.f;
  if (gs) g += gs[i];
  if (gd) g -= gd[i] / (sd * sd);
  gdisp[i] = c * g;
}

// ---------------------------------------------------------------- BackprojectDepth (layers.py:139-168)
__global__ void k_backproject(const float* __restrict__ depth, const float* __restrict__ invK,
                              float* __restrict__ out, int H, int W) {
  const int b = blockIdx.y, n = H * W;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const float* ik = invK + b * 16;
  const float x = (float)(p % W), y = (float)(p / W), d = depth[(size_t)b * n + p];
  float* o = out + (size_t)b * 4 * n + p;
#pragma unroll
  for (int k = 0; k < 3; ++k) o[(size_t)k * n] = d * fmaf(ik[k * 4 + 0], x, fmaf(ik[k * 4 + 1], y, ik[k * 4 + 2]));
  o[(size_t)3 * n] = 1.0f;
}
__global__ void k_backproject_bwd(const float* __restrict__ g, const float* __restrict__ invK,
                                  float* __restrict__ gdepth, int H, int W) {
  const int b = blockIdx.y, n = H * W;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const float* ik = invK + b * 16;
  const float x = (float)(p % W), y = (float)(p / W);
  const float* gi = g + (size_t)b * 4 * n + p;
  float a = 0.f;
#pragma unroll
  for (int k = 0; k < 3; ++k) a = fmaf(gi[(size_t)k * n], fmaf(ik[k * 4 + 0], x, fmaf(ik[k * 4 + 1], y, ik[k * 4 + 2])), a);
  gdepth[(size_t)b * n + p] = a;
}

// ---------------------------------------------------------------- Project3D (layers.py:171-193)
__device__ __forceinline__ void load_P(const float* K, const float* T, float P[3][4]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float a = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) a = fmaf(K[i * 4 + k], T[k * 4 + j], a);
      P[i][j] = a;
    }
}
__global__ void k_project3d(const float* __restrict__ pts, const float* __restrict__ K,
                            const float* __restrict__ T, float eps, float* __restrict__ out, int H, int W) {
  const int b = blockIdx.y, n = H * W;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  float P[3][4];
  load_P(K + b * 16, T + b * 16, P);
  const float* pi = pts + (size_t)b * 4 * n + p;
  const float X = pi[0], Y = pi[(size_t)n], Z = pi[(size_t)2 * n], Wc = pi[(size_t)3 * n];
  float c[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) c[i] = fmaf(P[i][0], X, fmaf(P[i][1], Y, fmaf(P[i][2], Z, P[i][3] * Wc)));
  const float den = c[2] + eps;
  const float u = c[0] / den, v = c[1] / den;
  float* o = out + ((size_t)b * n + p) * 2;
  o[0] = (u / (float)(W - 1) - 0.5f) * 2.0f;
  o[1] = (v / (float)(H - 1) - 0.5f) * 2.0f;
}
__global__ void k_project3d_bwd(const float* __restrict__ gpix, const float* __restrict__ pts,
                                const float* __restrict__ K, const float* __restrict__ T, float eps,
                                float* __restrict__ gpts, float* __restrict__ gT, int H, int W) {
  const int b = blockIdx.y, n = H * W;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  float P[3][4];
  load_P(K + b * 16, T + b * 16, P);
  float dP[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) dP[k] = 0.f;
  if (p < n) {
    const float* pi = pts + (size_t)b * 4 * n + p;
    const float Xh[4] = {pi[0], pi[(size_t)n], pi[(size_t)2 * n], pi[(size_t)3 * n]};
    float c[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) c[i] = fmaf(P[i][0], Xh[0], fmaf(P[i][1], Xh[1], fmaf(P[i][2], Xh[2], P[i][3] * Xh[3])));
    const float den = c[2] + eps, inv = 1.0f / den;
    const float u = c[0] * inv, v = c[1] * inv;
    const float du = gpix[((size_t)b * n + p) * 2 + 0] * 2.0f / (float)(W - 1);
    const float dv = gpix[((size_t)b * n + p) * 2 + 1] * 2.0f / (float)(H - 1);
    const float dc[3] = {du * inv, dv * inv, -(u * du + v * dv) * inv};
    if (gpts) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        gpts[(size_t)b * 4 * n + (size_t)j * n + p] = fmaf(P[0][j], dc[0], fmaf(P[1][j], dc[1], P[2][j] * dc[2]));
    }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) dP[i * 4 + j] = dc[i] * Xh[j];
  }
  if (gT) {
    // d T = K[:3,:]^T dP ; reduce dP over the block first
    __shared__ float red[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) {
      const float s = block_sum(dP[k]);
      if (threadIdx.x == 0) red[k] = s;
    }
    __syncthreads();
    if (threadIdx.x < 16) {
      const int k = threadIdx.x / 4, j = threadIdx.x % 4;
      const float* Kb = K + b * 16;
      float a = 0.f;
#pragma unroll
      for (int i = 0; i < 3; ++i) a = fmaf(Kb[i * 4 + k], red[i * 4 + j], a);
      atomicAdd(gT + b * 16 + threadIdx.x, a);
    }
  }
}

// ---------------------------------------------------------------- grid_sample border (trainer.py:384-387)
__device__ __forceinline__ float unnorm(float g, int size, int ac) {
  return ac ? (g + 1.0f) * 0.5f * (float)(size - 1) : ((g + 1.0f) * (float)size - 1.0f) * 0.5f;
}
__global__ void k_grid_sample(const float* __restrict__ img, const float* __restrict__ grid,
                              float* __restrict__ out, int C, int IH, int IW, int OH, int OW, int ac) {
  const int b = blockIdx.y, n = OH * OW;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const float gx = grid[((size_t)b * n + p) * 2], gy = grid[((size_t)b * n + p) * 2 + 1];
  const float ix = fminf(fmaxf(unnorm(gx, IW, ac), 0.f), (float)(IW - 1));
  const float iy = fminf(fmaxf(unnorm(gy, IH, ac), 0.f), (float)(IH - 1));
  const float fx = floorf(ix), fy = floorf(iy);
  const int x0 = (int)fx, y0 = (int)fy;
  const int x1 = min(x0 + 1, IW - 1), y1 = min(y0 + 1, IH - 1);
  const float wx = ix - fx, wy = iy - fy;
  for (int c = 0; c < C; ++c) {
    const float* im = img + ((size_t)b * C + c) * IH * IW;
    const float nw = im[y0 * IW + x0], ne = im[y0 * IW + x1], sw = im[y1 * IW + x0], se = im[y1 * IW + x1];
    const float top = fmaf(wx, ne - nw, nw), bot = fmaf(wx, se - sw, sw);
    out[((size_t)b * C + c) * n + p] = fmaf(wy, bot - top, top);
  }
}
__global__ void k_grid_sample_bwd(const float* __restrict__ go, const float* __restrict__ img,
                                  const float* __restrict__ grid, float* __restrict__ ggrid, int C,
                                  int IH, int IW, int OH, int OW, int ac) {
  const int b = blockIdx.y, n = OH * OW;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const float gx = grid[((size_t)b * n + p) * 2], gy = grid[((size_t)b * n + p) * 2 + 1];
  const float ux = unnorm(gx, IW, ac), uy = unnorm(gy, IH, ac);
  const float mx = (ux > 0.f && ux < (float)(IW - 1)) ? (ac ? 0.5f * (float)(IW - 1) : 0.5f * (float)IW) : 0.f;
  const float my = (uy > 0.f && uy < (float)(IH - 1)) ? (ac ? 0.5f * (float)(IH - 1) : 0.5f * (float)IH) : 0.f;
  const float ix = fminf(fmaxf(ux, 0.f), (float)(IW - 1)), iy = fminf(fmaxf(uy, 0.f), (float)(IH - 1));
  const float fx = floorf(ix), fy = floorf(iy);
  const int x0 = (int)fx, y0 = (int)fy;
  const int x1 = min(x0 + 1, IW - 1), y1 = min(y0 + 1, IH - 1);
  const float wx = ix - fx, wy = iy - fy;
  float dx = 0.f, dy = 0.f;
  for (int c = 0; c < C; ++c) {
    const float* im = img + ((size_t)b * C + c) * IH * IW;
    const float nw = im[y0 * IW + x0], ne = im[y0 * IW + x1], sw = im[y1 * IW + x0], se = im[y1 * IW + x1];
    const float g = go[((size_t)b * C + c) * n + p];
    const float dn = ne - nw, ds = se - sw;
    dx = fmaf(g, fmaf(wy, ds - dn, dn), dx);
    dy = fmaf(g, fmaf(wx, ds, sw) - fmaf(wx, dn, nw), dy);
  }
  ggrid[((size_t)b * n + p) * 2] = dx * mx;
  ggrid[((size_t)b * n + p) * 2 + 1] = dy * my;
}

// ---------------------------------------------------------------- SSIM (layers.py:218-248)
__device__ __forceinline__ int refl(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

// window statistics at (qx,qy); returns S and, when want, d(n/d)/dx_j = a + b x_j + c y_j scaled by -0.5*live
__device__ __forceinline__ float ssim_at(const float* __restrict__ x, const float* __restrict__ y, int H, int W,
                                         int qy, int qx, bool want, float& ca, float& cb, float& cc) {
  float sx = 0.f, sy = 0.f, sxx = 0.f, syy = 0.f, sxy = 0.f;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      const int o = refl(qy + dy, H) * W + refl(qx + dx, W);
      const float a = x[o], b = y[o];
      sx += a; sy += b; sxx = fmaf(a, a, sxx); syy = fmaf(b, b, syy); sxy = fmaf(a, b, sxy);
    }
  const float c1 = 0.0081f, c2 = 0.0729f;
  const float pxy = sx * sy, pp = fmaf(sx, sx, sy * sy);
  const float n1 = fmaf(2.f, pxy, c1), n2 = fmaf(2.f, fmaf(9.f, sxy, -pxy), c2);
  const float d1 = pp + c1, d2 = fmaf(9.f, sxx + syy, -pp) + c2;
  const float invD = 1.0f / (d1 * d2);
  const float Q = n1 * n2 * invD;
  const float raw = fmaf(-0.5f, Q, 0.5f);
  if (want) {
    const float k = (raw >= 0.f && raw <= 1.f) ? -0.5f : 0.f;
    const float QD = Q * invD;
    ca = k * 2.0f * (sy * (n2 - n1) * invD - sx * (d2 - d1) * QD);
    cb = k * -18.0f * d1 * QD;
    cc = k * 18.0f * n1 * invD;
  }
  return fminf(fmaxf(raw, 0.f), 1.f);
}
__global__ void k_ssim(const float* __restrict__ x, const float* __restrict__ y, float* __restrict__ out,
                       int H, int W) {
  const size_t plane = (size_t)H * W;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= H * W) return;
  const size_t base = (size_t)blockIdx.y * plane;
  float a, b, c;
  out[base + p] = ssim_at(x + base, y + base, H, W, p / W, p % W, false, a, b, c);
}
// grad wrt the first argument of ssim_at; call with (x,y) for grad_x and (y,x) for grad_y (SSIM is symmetric)
__global__ void k_ssim_bwd(const float* __restrict__ go, const float* __restrict__ x,
                           const float* __restrict__ y, float* __restrict__ gx, int H, int W) {
  const size_t plane = (size_t)H * W;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= H * W) return;
  const size_t base = (size_t)blockIdx.y * plane;
  const int jy = p / W, jx = p % W;
  const float xj = x[base + p], yj = y[base + p];
  float acc = 0.f;
  for (int dy = -1; dy <= 1; ++dy) {
    const int qy = jy + dy;
    if (qy < 0 || qy >= H) continue;
    const float my = 1.f + ((jy == 1 && qy == 0) ? 1.f : 0.f) + ((jy == H - 2 && qy == H - 1) ? 1.f : 0.f);
    for (int dx = -1; dx <= 1; ++dx) {
      const int qx = jx + dx;
      if (qx < 0 || qx >= W) continue;
      const float mx = 1.f + ((jx == 1 && qx == 0) ? 1.f : 0.f) + ((jx == W - 2 && qx == W - 1) ? 1.f : 0.f);
      float a, b, c;
      ssim_at(x + base, y + base, H, W, qy, qx, true, a, b, c);
      acc = fmaf(my * mx * go[base + (size_t)qy * W + qx], fmaf(b, xj, fmaf(c, yj, a)), acc);
    }
  }
  gx[base + p] = acc;
}

// ---------------------------------------------------------------- get_smooth_loss (layers.py:202-215)
__device__ __forceinline__ float edge_w(const float* __restrict__ img, int C, size_t plane, size_t pa, size_t pb) {
  float g = 0.f;
  for (int c = 0; c < C; ++c) g += fabsf(img[c * plane + pa] - img[c * plane + pb]);
  return expf(-(g / (float)C));
}
__global__ void k_smooth_fwd(const float* __restrict__ disp, const float* __restrict__ img, double* acc,
                             int C, int H, int W) {
  const int b = blockIdx.y, n = H * W;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  float ex = 0.f, ey = 0.f;
  if (p < n) {
    const float* d = disp + (size_t)b * n;
    const float* im = img + (size_t)b * C * n;
    const int x = p % W, y = p / W;
    if (x + 1 < W) ex = fabsf(d[p] - d[p + 1]) * edge_w(im, C, n, p, p + 1);
    if (y + 1 < H) ey = fabsf(d[p] - d[p + W]) * edge_w(im, C, n, p, p + W);
  }
  ex = block_sum(ex);
  ey = block_sum(ey);
  if (threadIdx.x == 0) { atomicAdd(acc, (double)ex); atomicAdd(acc + 1, (double)ey); }
}
__global__ void k_smooth_finish(const double* acc, float* loss, double nx, double ny) {
  loss[0] = (float)(acc[0] / nx + acc[1] / ny);
}
__global__ void k_smooth_bwd(const float* __restrict__ gl, const float* __restrict__ disp,
                             const float* __restrict__ img, float* __restrict__ gd, int C, int H, int W,
                             float inx, float iny) {
  const int b = blockIdx.y, n = H * W;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const float* d = disp + (size_t)b * n;
  const float* im = img + (size_t)b * C * n;
  const int x = p % W, y = p / W;
  auto sg = [](float v) { return v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f); };
  float g = 0.f;
  if (x + 1 < W) g += inx * sg(d[p] - d[p + 1]) * edge_w(im, C, n, p, p + 1);
  if (x > 0) g -= inx * sg(d[p - 1] - d[p]) * edge_w(im, C, n, p - 1, p);
  if (y + 1 < H) g += iny * sg(d[p] - d[p + W]) * edge_w(im, C, n, p, p + W);
  if (y > 0) g -= iny * sg(d[p - W] - d[p]) * edge_w(im, C, n, p - W, p);
  gd[(size_t)b * n + p] = g * gl[0];
}

// ---------------------------------------------------------------- pose -> 4x4 (layers.py:28-103)
// (the per-sample arithmetic lives in md2_core.cuh: the fused call builds T from the pose leaves itself)
__global__ void k_pose_to_matrix(const float* __restrict__ aa, const float* __restrict__ tr, int invert,
                                 float* __restrict__ T, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  md2::pose_to_matrix(aa + b * 3, tr + b * 3, invert, T + b * 16);
}
__global__ void k_pose_to_matrix_bwd(const float* __restrict__ gT, const float* __restrict__ aa,
                                     const float* __restrict__ tr, int invert, float* __restrict__ gaa,
                                     float* __restrict__ gtr, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  md2::pose_to_matrix_backward(gT + b * 16, aa + b * 3, tr + b * 3, invert, gaa + b * 3, gtr + b * 3);
}

}  // namespace

struct ScaleArgs {
  const float* src[MD2_MAX_SCALE_TENSORS];
  float* dst[MD2_MAX_SCALE_TENSORS];
  long long start[MD2_MAX_SCALE_TENSORS + 1];
  long long numel[MD2_MAX_SCALE_TENSORS];
  int n;
};
__global__ void k_scale_tensors(ScaleArgs a, const float* __restrict__ scale) {
  const long long q = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;      // 4 consecutive elements per thread
  if (q >= a.start[a.n]) return;
  int i = 0;
  while (i + 1 < a.n && q >= a.start[i + 1]) ++i;
  const long long j = q - a.start[i];
  const float g = __ldg(scale);
  const float* s = a.src[i];
  float* d = a.dst[i];
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (j + k < a.numel[i]) d[j + k] = __ldg(s + j + k) * g;
}

// md2_scale_tensors with a destination type per tensor: the fp32 product, rounded once (round-to-nearest-even; an
// overflow rounds to +-inf, which GradScaler's found-inf check relies on)
struct ScaleTypedArgs {
  const float* src[MD2_MAX_SCALE_TENSORS];
  void* dst[MD2_MAX_SCALE_TENSORS];
  long long start[MD2_MAX_SCALE_TENSORS + 1];
  long long numel[MD2_MAX_SCALE_TENSORS];
  int dtype[MD2_MAX_SCALE_TENSORS];
  int n;
};
__global__ void k_scale_tensors_typed(ScaleTypedArgs a, const float* __restrict__ scale) {
  const long long q = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (q >= a.start[a.n]) return;
  int i = 0;
  while (i + 1 < a.n && q >= a.start[i + 1]) ++i;
  const long long j = q - a.start[i];
  const float g = __ldg(scale);
  const float* s = a.src[i];
  const int dt = a.dtype[i];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (j + k >= a.numel[i]) break;
    const float v = __ldg(s + j + k) * g;
    if (dt == MD2_DTYPE_BF16) ((__nv_bfloat16*)a.dst[i])[j + k] = __float2bfloat16_rn(v);
    else if (dt == MD2_DTYPE_F16) ((__half*)a.dst[i])[j + k] = __float2half_rn(v);
    else ((float*)a.dst[i])[j + k] = v;
  }
}

extern "C" {

int md2_disp_to_depth(const float* disp, float min_depth, float max_depth, float* scaled_disp, float* depth,
                      long long n, void* stream) {
  if (!disp || n < 0 || !(min_depth > 0.f) || !(max_depth > min_depth)) return MD2_ERR_INVALID_ARGUMENT;
  if (n == 0) return MD2_OK;
  const double lo = 1.0 / max_depth, hi = 1.0 / min_depth;
  k_disp_to_depth<<<blocks_for(n), kT, 0, (cudaStream_t)stream>>>(disp, (float)lo, (float)(hi - lo), scaled_disp, depth, n);
  return rc(cudaGetLastError());
}
int md2_disp_to_depth_backward(const float* disp, float min_depth, float max_depth, const float* grad_scaled,
                               const float* grad_depth, float* grad_disp, long long n, void* stream) {
  if (!disp || !grad_disp || n < 0) return MD2_ERR_INVALID_ARGUMENT;
  if (n == 0) return MD2_OK;
  const double lo = 1.0 / max_depth, hi = 1.0 / min_depth;
  k_disp_to_depth_bwd<<<blocks_for(n), kT, 0, (cudaStream_t)stream>>>(disp, (float)lo, (float)(hi - lo), grad_scaled, grad_depth, grad_disp, n);
  return rc(cudaGetLastError());
}

int md2_backproject_depth(const float* depth, const float* inv_K, float* cam_points, int batch, int height,
                          int width, void* stream) {
  if (!depth || !inv_K || !cam_points || batch < 1 || height < 1 || width < 1) return MD2_ERR_INVALID_ARGUMENT;
  dim3 grid(blocks_for((long long)height * width), batch);
  k_backproject<<<grid, kT, 0, (cudaStream_t)stream>>>(depth, inv_K, cam_points, height, width);
  return rc(cudaGetLastError());
}
int md2_backproject_depth_backward(const float* grad_cam_points, const float* inv_K, float* grad_depth,
                                   int batch, int height, int width, void* stream) {
  if (!grad_cam_points || !inv_K || !grad_depth || batch < 1 || height < 1 || width < 1) return MD2_ERR_INVALID_ARGUMENT;
  dim3 grid(blocks_for((long long)height * width), batch);
  k_backproject_bwd<<<grid, kT, 0, (cudaStream_t)stream>>>(grad_cam_points, inv_K, grad_depth, height, width);
  return rc(cudaGetLastError());
}

int md2_project3d(const float* points, const float* K, const float* T, float eps, float* pix_coords,
                  int batch, int height, int width, void* stream) {
  if (!points || !K || !T || !pix_coords || batch < 1 || height < 2 || width < 2) return MD2_ERR_INVALID_ARGUMENT;
  dim3 grid(blocks_for((long long)height * width), batch);
  k_project3d<<<grid, kT, 0, (cudaStream_t)stream>>>(points, K, T, eps, pix_coords, height, width);
  return rc(cudaGetLastError());
}
int md2_project3d_backward(const float* grad_pix, const float* points, const float* K, const float* T,
                           float eps, float* grad_points, float* grad_T, int batch, int height, int width,
                           void* stream) {
  if (!grad_pix || !points || !K || !T || batch < 1 || height < 2 || width < 2) return MD2_ERR_INVALID_ARGUMENT;
  cudaStream_t s = (cudaStream_t)stream;
  if (grad_T) {
    cudaError_t e = cudaMemsetAsync(grad_T, 0, sizeof(float) * 16 * batch, s);
    if (e != cudaSuccess) return MD2_ERR_CUDA;
  }
  dim3 grid(blocks_for((long long)height * width), batch);
  k_project3d_bwd<<<grid, kT, 0, s>>>(grad_pix, points, K, T, eps, grad_points, grad_T, height, width);
  return rc(cudaGetLastError());
}

int md2_grid_sample_border(const float* img, const float* grid, float* out, int batch, int channels, int in_h,
                           int in_w, int out_h, int out_w, int align_corners, void* stream) {
  if (!img || !grid || !out || batch < 1 || channels < 1 || in_h < 1 || in_w < 1 || out_h < 1 || out_w < 1)
    return MD2_ERR_INVALID_ARGUMENT;
  dim3 g(blocks_for((long long)out_h * out_w), batch);
  k_grid_sample<<<g, kT, 0, (cudaStream_t)stream>>>(img, grid, out, channels, in_h, in_w, out_h, out_w, align_corners);
  return rc(cudaGetLastError());
}
int md2_grid_sample_border_backward(const float* grad_out, const float* img, const float* grid, float* grad_grid,
                                    int batch, int channels, int in_h, int in_w, int out_h, int out_w,
                                    int align_corners, void* stream) {
  if (!grad_out || !img || !grid || !grad_grid || batch < 1 || channels < 1) return MD2_ERR_INVALID_ARGUMENT;
  dim3 g(blocks_for((long long)out_h * out_w), batch);
  k_grid_sample_bwd<<<g, kT, 0, (cudaStream_t)stream>>>(grad_out, img, grid, grad_grid, channels, in_h, in_w, out_h, out_w, align_corners);
  return rc(cudaGetLastError());
}

int md2_ssim(const float* x, const float* y, float* out, int batch, int channels, int height, int width,
             void* stream) {
  if (!x || !y || !out || batch < 1 || channels < 1 || height < 2 || width < 2) return MD2_ERR_INVALID_ARGUMENT;
  dim3 g(blocks_for((long long)height * width), batch * channels);
  k_ssim<<<g, kT, 0, (cudaStream_t)stream>>>(x, y, out, height, width);
  return rc(cudaGetLastError());
}
int md2_ssim_backward(const float* grad_out, const float* x, const float* y, float* grad_x, float* grad_y,
                      int batch, int channels, int height, int width, void* stream) {
  if (!grad_out || !x || !y || batch < 1 || channels < 1 || height < 2 || width < 2) return MD2_ERR_INVALID_ARGUMENT;
  dim3 g(blocks_for((long long)height * width), batch * channels);
  if (grad_x) k_ssim_bwd<<<g, kT, 0, (cudaStream_t)stream>>>(grad_out, x, y, grad_x, height, width);
  if (grad_y) k_ssim_bwd<<<g, kT, 0, (cudaStream_t)stream>>>(grad_out, y, x, grad_y, height, width);
  return rc(cudaGetLastError());
}

int md2_smooth_loss(const float* disp, const float* img, float* loss, void* scratch16, int batch, int channels,
                    int height, int width, void* stream) {
  if (!disp || !img || !loss || !scratch16 || batch < 1 || channels < 1 || height < 2 || width < 2)
    return MD2_ERR_INVALID_ARGUMENT;
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaMemsetAsync(scratch16, 0, 16, s) != cudaSuccess) return MD2_ERR_CUDA;
  dim3 g(blocks_for((long long)height * width), batch);
  k_smooth_fwd<<<g, kT, 0, s>>>(disp, img, (double*)scratch16, channels, height, width);
  k_smooth_finish<<<1, 1, 0, s>>>((const double*)scratch16, loss, (double)batch * height * (width - 1),
                                  (double)batch * (height - 1) * width);
  return rc(cudaGetLastError());
}
int md2_smooth_loss_backward(const float* grad_loss, const float* disp, const float* img, float* grad_disp,
                             int batch, int channels, int height, int width, void* stream) {
  if (!grad_loss || !disp || !img || !grad_disp || batch < 1 || channels < 1 || height < 2 || width < 2)
    return MD2_ERR_INVALID_ARGUMENT;
  dim3 g(blocks_for((long long)height * width), batch);
  k_smooth_bwd<<<g, kT, 0, (cudaStream_t)stream>>>(grad_loss, disp, img, grad_disp, channels, height, width,
                                                   1.0f / ((float)batch * height * (width - 1)),
                                                   1.0f / ((float)batch * (height - 1) * width));
  return rc(cudaGetLastError());
}

int md2_pose_to_matrix(const float* axisangle, const float* translation, int invert, float* T, int batch,
                       void* stream) {
  if (!axisangle || !translation || !T || batch < 1) return MD2_ERR_INVALID_ARGUMENT;
  k_pose_to_matrix<<<blocks_for(batch), kT, 0, (cudaStream_t)stream>>>(axisangle, translation, invert, T, batch);
  return rc(cudaGetLastError());
}
int md2_pose_to_matrix_backward(const float* grad_T, const float* axisangle, const float* translation, int invert,
                                float* grad_axisangle, float* grad_translation, int batch, void* stream) {
  if (!grad_T || !axisangle || !translation || !grad_axisangle || !grad_translation || batch < 1)
    return MD2_ERR_INVALID_ARGUMENT;
  k_pose_to_matrix_bwd<<<blocks_for(batch), kT, 0, (cudaStream_t)stream>>>(grad_T, axisangle, translation, invert,
                                                                         grad_axisangle, grad_translation, batch);
  return rc(cudaGetLastError());
}

/* autograd glue of the fused call: dst[i] = src[i] * (*scale) for up to MD2_MAX_SCALE_TENSORS tensors in ONE launch
 * (the backward of the torch.autograd.Function multiplies every stored gradient by the incoming scalar gradient). */
int md2_scale_tensors(int n_tensors, const float* const* src, float* const* dst, const long long* numel,
                      const float* scale, void* stream) {
  if (n_tensors < 1 || n_tensors > MD2_MAX_SCALE_TENSORS || !src || !dst || !numel || !scale) return MD2_ERR_INVALID_ARGUMENT;
  ScaleArgs a;
  long long total = 0;
  for (int i = 0; i < n_tensors; ++i) {
    if (!src[i] || !dst[i] || numel[i] < 0) return MD2_ERR_INVALID_ARGUMENT;
    a.src[i] = src[i]; a.dst[i] = dst[i]; a.start[i] = total;
    total += (numel[i] + 3) / 4 * 4;          // every tensor starts on a multiple of 4 of the flat index space
  }
  a.start[n_tensors] = total;
  a.n = n_tensors;
  for (int i = 0; i < n_tensors; ++i) a.numel[i] = numel[i];
  if (total == 0) return MD2_OK;
  const long long threads = total / 4;
  k_scale_tensors<<<(unsigned)((threads + kT - 1) / kT), kT, 0, (cudaStream_t)stream>>>(a, scale);
  return rc(cudaGetLastError());
}

int md2_scale_tensors_typed(int n_tensors, const float* const* src, void* const* dst, const int* dst_dtype,
                            const long long* numel, const float* scale, void* stream) {
  if (n_tensors < 1 || n_tensors > MD2_MAX_SCALE_TENSORS || !src || !dst || !dst_dtype || !numel || !scale)
    return MD2_ERR_INVALID_ARGUMENT;
  ScaleTypedArgs a;
  long long total = 0;
  for (int i = 0; i < n_tensors; ++i) {
    const int d = dst_dtype[i];
    if (!src[i] || !dst[i] || numel[i] < 0) return MD2_ERR_INVALID_ARGUMENT;
    if (d != MD2_DTYPE_F32 && d != MD2_DTYPE_BF16 && d != MD2_DTYPE_F16) return MD2_ERR_INVALID_ARGUMENT;
    a.src[i] = src[i]; a.dst[i] = dst[i]; a.dtype[i] = d; a.start[i] = total;
    total += (numel[i] + 3) / 4 * 4;
  }
  a.start[n_tensors] = total;
  a.n = n_tensors;
  for (int i = 0; i < n_tensors; ++i) a.numel[i] = numel[i];
  if (total == 0) return MD2_OK;
  const long long threads = total / 4;
  k_scale_tensors_typed<<<(unsigned)((threads + kT - 1) / kT), kT, 0, (cudaStream_t)stream>>>(a, scale);
  return rc(cudaGetLastError());
}

}  // extern "C"
