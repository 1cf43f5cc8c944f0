// md2_head.cu - decoder tail that feeds the loss path (SURVEY.md 8f-4): the disparity head of DepthDecoder,
//   outputs[("disp", s)] = sigmoid(Conv3x3(num_ch_dec[s] -> 1)(x))       /root/reference/networks/depth_decoder.py:60-63
// with Conv3x3 = ReflectionPad2d(1) + Conv2d(C, 1, 3) (/root/reference/layers.py:119-136), at 4 scales
// (C = 16, 32, 64, 128 at H, H/2, H/4, H/8).  One output channel is the worst case for a library convolution
// (no reuse across output channels: pure bandwidth); here pad, convolution, bias and sigmoid are one pass that reads the
// feature map once, and the backward is two passes (input gradient in gather form, weight gradient as a reduction).
// The feature-map side (x, disp, grad_disp, grad_x) is a template parameter: fp32, or bf16 / fp16 read at 2 bytes a value,
// widened exactly and rounded once on the way out; weights, bias and the arithmetic are fp32 in every instantiation.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/md2_loss.h"

namespace {

constexpr int kT = 256;

__device__ __forceinline__ int reflect1(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

__device__ __forceinline__ float ldf(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldf(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
__device__ __forceinline__ float ldf(const __half* p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ void stf(float* p, float v) { *p = v; }
__device__ __forceinline__ void stf(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void stf(__half* p, float v) { *p = __float2half_rn(v); }

// forward: one thread per output pixel, weights in shared memory
template <typename T>
__global__ void __launch_bounds__(kT) k_dispconv_fwd(const T* __restrict__ x, const float* __restrict__ w,
                                                     const float* __restrict__ bias, T* __restrict__ disp,
                                                     int B, int C, int H, int W) {
  extern __shared__ float ws[];                 // C x 9
  for (int i = threadIdx.x; i < C * 9; i += blockDim.x) ws[i] = __ldg(w + i);
  __syncthreads();
  const int plane = H * W;
  const long long n = (long long)B * plane;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int b = (int)(i / plane), p = (int)(i - (long long)b * plane);
  const int y = p / W, xx = p - y * W;
  int off[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) off[k] = reflect1(y + k / 3 - 1, H) * W + reflect1(xx + k % 3 - 1, W);
  const T* xb = x + (size_t)b * C * plane;
  float acc = __ldg(bias);
  for (int c = 0; c < C; ++c) {
    const T* xc = xb + (size_t)c * plane;
    const float* wc = ws + c * 9;
#pragma unroll
    for (int k = 0; k < 9; ++k) acc = fmaf(ldf(xc + off[k]), wc[k], acc);
  }
  stf(disp + i, 1.0f / (1.0f + __expf(-acc)));
}

// grad of the pre-activation: g * s * (1 - s)
template <typename T>
__device__ __forceinline__ float gpre(const T* __restrict__ gd, const T* __restrict__ disp, size_t i) {
  const float s = ldf(disp + i);
  return ldf(gd + i) * s * (1.0f - s);
}

// input gradient, gather form.  Padded coordinate set that maps onto index i of a reflect-padded axis of length n:
// {i}, plus {-1} when i == 1 and {n} when i == n-2.
template <typename T>
__global__ void __launch_bounds__(kT) k_dispconv_bwd_input(const T* __restrict__ gd, const T* __restrict__ disp,
                                                           const float* __restrict__ w, T* __restrict__ gx,
                                                           int B, int C, int H, int W) {
  extern __shared__ float ws[];
  for (int i = threadIdx.x; i < C * 9; i += blockDim.x) ws[i] = __ldg(w + i);
  __syncthreads();
  const int plane = H * W;
  const long long n = (long long)B * plane;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int b = (int)(i / plane), p = (int)(i - (long long)b * plane);
  const int y = p / W, xx = p - y * W;
  int py[3], px[3], ny = 0, nx = 0;
  py[ny++] = y; if (y == 1) py[ny++] = -1; if (y == H - 2) py[ny++] = H;
  px[nx++] = xx; if (xx == 1) px[nx++] = -1; if (xx == W - 2) px[nx++] = W;
  // contributions: output pixel q = (pady - ky, padx - kx) with tap k; at most 4 x 9 of them
  float g[36];
  int kk[36];
  int m = 0;
  for (int a = 0; a < ny; ++a)
    for (int c = 0; c < nx; ++c)
      for (int k = 0; k < 9; ++k) {
        const int qy = py[a] - (k / 3 - 1), qx = px[c] - (k % 3 - 1);
        if (qy < 0 || qy >= H || qx < 0 || qx >= W) continue;
        g[m] = gpre(gd, disp, (size_t)b * plane + (size_t)qy * W + qx);
        kk[m] = k;
        ++m;
      }
  T* gb = gx + (size_t)b * C * plane + p;
  for (int c = 0; c < C; ++c) {
    const float* wc = ws + c * 9;
    float acc = 0.f;
    for (int j = 0; j < m; ++j) acc = fmaf(g[j], wc[kk[j]], acc);
    stf(gb + (size_t)c * plane, acc);
  }
}

// weight / bias gradient: block = (channel c, chunk of pixels); 9 sums per thread, block reduction, one atomic per sum
template <typename T>
__global__ void __launch_bounds__(kT) k_dispconv_bwd_weight(const T* __restrict__ gd, const T* __restrict__ disp,
                                                            const T* __restrict__ x, float* __restrict__ gw,
                                                            float* __restrict__ gbias, int B, int C, int H, int W) {
  const int c = blockIdx.y;
  const int plane = H * W;
  const long long n = (long long)B * plane;
  float acc[10];
#pragma unroll
  for (int k = 0; k < 10; ++k) acc[k] = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / plane), p = (int)(i - (long long)b * plane);
    const int y = p / W, xx = p - y * W;
    const float g = gpre(gd, disp, (size_t)i);
    const T* xc = x + ((size_t)b * C + c) * plane;
#pragma unroll
    for (int k = 0; k < 9; ++k)
      acc[k] = fmaf(g, ldf(xc + reflect1(y + k / 3 - 1, H) * W + reflect1(xx + k % 3 - 1, W)), acc[k]);
    acc[9] += g;
  }
  __shared__ float red[10][kT / 32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 10; ++k) {
    float v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[k][wid] = v;
  }
  __syncthreads();
  if (threadIdx.x < 10) {
    float v = 0.f;
    for (int j = 0; j < kT / 32; ++j) v += red[threadIdx.x][j];
    if (threadIdx.x < 9) atomicAdd(gw + c * 9 + threadIdx.x, v);
    else if (c == 0 && gbias) atomicAdd(gbias, v);
  }
}

int rc(cudaError_t e) { return e == cudaSuccess ? MD2_OK : MD2_ERR_CUDA; }

template <typename T>
int head_fwd(const T* x, const float* weight, const float* bias, T* disp, int batch, int channels, int height, int width,
             void* stream) {
  if (!x || !weight || !bias || !disp || batch < 1 || channels < 1 || height < 2 || width < 2) return MD2_ERR_INVALID_ARGUMENT;
  if ((size_t)channels * 9 * sizeof(float) > 48 * 1024) return MD2_ERR_UNSUPPORTED;
  const long long n = (long long)batch * height * width;
  k_dispconv_fwd<T><<<(unsigned)((n + kT - 1) / kT), kT, channels * 9 * sizeof(float), (cudaStream_t)stream>>>(
      x, weight, bias, disp, batch, channels, height, width);
  return rc(cudaGetLastError());
}

template <typename T>
int head_bwd(const T* grad_disp, const T* disp, const T* x, const float* weight, T* grad_x, float* grad_weight,
             float* grad_bias, int batch, int channels, int height, int width, void* stream) {
  if (!grad_disp || !disp || !x || !weight || batch < 1 || channels < 1 || height < 2 || width < 2) return MD2_ERR_INVALID_ARGUMENT;
  if ((size_t)channels * 9 * sizeof(float) > 48 * 1024) return MD2_ERR_UNSUPPORTED;
  cudaStream_t s = (cudaStream_t)stream;
  const long long n = (long long)batch * height * width;
  if (grad_x)
    k_dispconv_bwd_input<T><<<(unsigned)((n + kT - 1) / kT), kT, channels * 9 * sizeof(float), s>>>(
        grad_disp, disp, weight, grad_x, batch, channels, height, width);
  if (grad_weight) {
    if (cudaMemsetAsync(grad_weight, 0, (size_t)channels * 9 * sizeof(float), s) != cudaSuccess) return MD2_ERR_CUDA;
    if (grad_bias && cudaMemsetAsync(grad_bias, 0, sizeof(float), s) != cudaSuccess) return MD2_ERR_CUDA;
    long long chunks = (n + (long long)kT * 16 - 1) / ((long long)kT * 16);
    if (chunks > 592) chunks = 592;
    if (chunks < 1) chunks = 1;
    dim3 grid((unsigned)chunks, (unsigned)channels);
    k_dispconv_bwd_weight<T><<<grid, kT, 0, s>>>(grad_disp, disp, x, grad_weight, grad_bias, batch, channels, height, width);
  }
  return rc(cudaGetLastError());
}

}  // namespace

extern "C" {

int md2_dispconv_sigmoid(const float* x, const float* weight, const float* bias, float* disp, int batch, int channels,
                         int height, int width, void* stream) {
  return head_fwd<float>(x, weight, bias, disp, batch, channels, height, width, stream);
}

int md2_dispconv_sigmoid_backward(const float* grad_disp, const float* disp, const float* x, const float* weight,
                                  float* grad_x, float* grad_weight, float* grad_bias, int batch, int channels, int height,
                                  int width, void* stream) {
  return head_bwd<float>(grad_disp, disp, x, weight, grad_x, grad_weight, grad_bias, batch, channels, height, width, stream);
}

int md2_dispconv_sigmoid_typed(const void* x, const float* weight, const float* bias, void* disp, int dtype, int batch,
                               int channels, int height, int width, void* stream) {
  switch (dtype) {
    case MD2_DTYPE_F32:
      return head_fwd<float>((const float*)x, weight, bias, (float*)disp, batch, channels, height, width, stream);
    case MD2_DTYPE_BF16:
      return head_fwd<__nv_bfloat16>((const __nv_bfloat16*)x, weight, bias, (__nv_bfloat16*)disp, batch, channels,
                                     height, width, stream);
    case MD2_DTYPE_F16:
      return head_fwd<__half>((const __half*)x, weight, bias, (__half*)disp, batch, channels, height, width, stream);
    default: return MD2_ERR_INVALID_ARGUMENT;
  }
}

int md2_dispconv_sigmoid_backward_typed(const void* grad_disp, const void* disp, const void* x, const float* weight,
                                        void* grad_x, float* grad_weight, float* grad_bias, int dtype, int batch,
                                        int channels, int height, int width, void* stream) {
  switch (dtype) {
    case MD2_DTYPE_F32:
      return head_bwd<float>((const float*)grad_disp, (const float*)disp, (const float*)x, weight, (float*)grad_x,
                             grad_weight, grad_bias, batch, channels, height, width, stream);
    case MD2_DTYPE_BF16: {
      typedef __nv_bfloat16 T;
      return head_bwd<T>((const T*)grad_disp, (const T*)disp, (const T*)x, weight, (T*)grad_x, grad_weight, grad_bias,
                         batch, channels, height, width, stream);
    }
    case MD2_DTYPE_F16: {
      typedef __half T;
      return head_bwd<T>((const T*)grad_disp, (const T*)disp, (const T*)x, weight, (T*)grad_x, grad_weight, grad_bias,
                         batch, channels, height, width, stream);
    }
    default: return MD2_ERR_INVALID_ARGUMENT;
  }
}

}  // extern "C"
