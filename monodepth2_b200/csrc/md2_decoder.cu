// md2_decoder.cu - the data movement in front of every ConvBlock of DepthDecoder (SURVEY.md 8f-4, second part):
//   out = ReflectionPad2d(1)(cat([nearest_up(x, up), skip], dim=1))    /root/reference/networks/depth_decoder.py:48-65,
//                                                                      layers.py:106-136 (Conv3x3 pad), 196-199 (upsample)
// x (B,Cx,h,w), skip (B,Cs,up*h,up*w) or none (Cs = 0), out (B,Cx+Cs,up*h+2,up*w+2).  The reference runs this as
// upsample + torch.cat + ReflectionPad2d (three launches, two intermediate tensors); here it is one producer pass that
// reads x and skip once and writes the padded input of the convolution.
//
// Forward is pure data movement: every dtype is bit-identical to torch's chain.  Backward is in gather form: each
// thread owns elements of grad_x / grad_skip and sums the padded positions that were read from them, so there are no
// atomics and the result is the same from run to run (ATen's reflection_pad2d_backward is an atomic scatter, refused
// by torch.use_deterministic_algorithms).
//   fold(r, q)  = padded (r+1, q+1), then its mirrors: row 0 when r == 1, row H2+1 when r == H2-2, the same for columns
//                 (own position first, summed from 0.0f; 1 to 4 terms, 3 per axis when that axis is 3 long)
//   grad_skip   = fold(r, q)
//   grad_x      = sum over the up x up children of fold, row-major, from 0.0f  (ATen's upsample_nearest2d_backward)
// Where every fold has at most two terms this is bitwise torch's fp32 chain (its zero-initialised atomic adds of two
// terms are exact in any order).  Arithmetic is fp32; bf16 / fp16 values are widened exactly and every result is
// rounded once to nearest-even.
//
// Each thread handles one 16-byte chunk of the array it writes (4 fp32 or 8 bf16 / fp16 values) and stores it with one
// vector store when the array is 16-byte aligned; chunks are aligned to the array, not to rows, because a padded row of
// up*w+2 values is often not a multiple of 16 bytes.  A chunk may span rows (small planes), which the loops handle.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <limits.h>
#include <stdint.h>

#include "../../include/md2_loss.h"

namespace {

constexpr int kT = 256;

__device__ __forceinline__ int reflect1(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

__device__ __forceinline__ float ldf(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldf(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
__device__ __forceinline__ float ldf(const __half* p) { return __half2float(__ldg(p)); }
template <typename T> __device__ __forceinline__ T fromf(float v);
template <> __device__ __forceinline__ float fromf<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 fromf<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half fromf<__half>(float v) { return __float2half_rn(v); }

// one 16-byte chunk of T
template <typename T>
struct alignas(16) Chunk {
  static constexpr int V = 16 / sizeof(T);
  T v[V];
};

// writes the first n (<= V) values of c at p: one vector store for a full, aligned chunk
template <typename T>
__device__ __forceinline__ void store_chunk(T* p, const Chunk<T>& c, int n, bool aligned) {
  if (aligned && n == Chunk<T>::V) {
    *reinterpret_cast<uint4*>(p) = *reinterpret_cast<const uint4*>(&c);
  } else {
    for (int k = 0; k < n; ++k) p[k] = c.v[k];
  }
}

struct Dims {
  int Cx, Cs, C;       // channels of x, skip, out
  int h, w;            // x
  int H2, W2;          // up-sampled = skip
  int Ho, Wo;          // out = H2 + 2, W2 + 2
  int up_shift;        // log2(up)
};

// -------------------------------------------------------------------------------------------------- forward
// Source row of output row `row` (= (b*C + c)*Ho + Y): a pointer to the row of x or skip it reads, and the shift that
// maps an up-sampled column onto it (log2(up) for x, 0 for skip).
template <typename T>
__device__ __forceinline__ const T* fwd_src_row(const T* __restrict__ x, const T* __restrict__ skip, const Dims& d,
                                                unsigned row, int* shift) {
  const unsigned plane = row / (unsigned)d.Ho;
  const int Y = (int)(row - plane * (unsigned)d.Ho);
  const unsigned b = plane / (unsigned)d.C;
  const int c = (int)(plane - b * (unsigned)d.C);
  const int r = reflect1(Y - 1, d.H2);
  if (c < d.Cx) {
    *shift = d.up_shift;
    return x + ((size_t)(b * (unsigned)d.Cx + (unsigned)c) * d.h + (r >> d.up_shift)) * d.w;
  }
  *shift = 0;
  return skip + ((size_t)(b * (unsigned)d.Cs + (unsigned)(c - d.Cx)) * d.H2 + r) * d.W2;
}

template <typename T>
__global__ void __launch_bounds__(kT) k_upcat_pad(const T* __restrict__ x, const T* __restrict__ skip,
                                                  T* __restrict__ out, Dims d, unsigned n, bool aligned) {
  constexpr int V = Chunk<T>::V;
  const unsigned chunk = blockIdx.x * (unsigned)blockDim.x + threadIdx.x;
  const unsigned e0 = chunk * (unsigned)V;
  if (e0 >= n) return;
  const int cnt = n - e0 < (unsigned)V ? (int)(n - e0) : V;
  unsigned row = e0 / (unsigned)d.Wo;
  int X = (int)(e0 - row * (unsigned)d.Wo);
  int shift;
  const T* src = fwd_src_row(x, skip, d, row, &shift);
  Chunk<T> c;
#pragma unroll
  for (int k = 0; k < V; ++k) {
    if (k < cnt) {
      if (X == d.Wo) {
        X = 0;
        src = fwd_src_row(x, skip, d, ++row, &shift);
      }
      c.v[k] = src[reflect1(X - 1, d.W2) >> shift];
      ++X;
    }
  }
  store_chunk(out + e0, c, cnt, aligned);
}

// -------------------------------------------------------------------------------------------------- backward
// fold(r, q) of one grad_out plane `g` (row stride Wo), summed from 0.0f.  The padded rows (columns) that fold onto
// up-sampled index r of an axis of length n are r+1, then 0 if r == 1, then n+1 if r == n-2; the terms are taken row
// by row in that order and, within a row, column by column in that order, so the own position comes first.
template <typename T>
__device__ __forceinline__ float fold_row(const T* __restrict__ p, int q, bool mx0, bool mx1, int W2, float acc) {
  acc += ldf(p + q + 1);
  if (mx0) acc += ldf(p);
  if (mx1) acc += ldf(p + W2 + 1);
  return acc;
}

template <typename T>
__device__ __forceinline__ float fold(const T* __restrict__ g, int r, int q, const Dims& d) {
  const bool mx0 = q == 1, mx1 = q == d.W2 - 2;
  float acc = fold_row(g + (size_t)(r + 1) * d.Wo, q, mx0, mx1, d.W2, 0.0f);
  if (r == 1) acc = fold_row(g, q, mx0, mx1, d.W2, acc);
  if (r == d.H2 - 2) acc = fold_row(g + (size_t)(d.H2 + 1) * d.Wo, q, mx0, mx1, d.W2, acc);
  return acc;
}

// grad_out plane of grad_x row `row` (= (b*Cx + c)*h + i); sets i
template <typename T>
__device__ __forceinline__ const T* bwd_x_plane(const T* __restrict__ gout, const Dims& d, unsigned row, int* i) {
  const unsigned plane = row / (unsigned)d.h;
  *i = (int)(row - plane * (unsigned)d.h);
  const unsigned b = plane / (unsigned)d.Cx;
  const unsigned ch = plane - b * (unsigned)d.Cx;
  return gout + (size_t)(b * (unsigned)d.C + ch) * ((size_t)d.Ho * d.Wo);
}

// grad_out plane of grad_skip row `row` (= (b*Cs + c)*H2 + r); sets r
template <typename T>
__device__ __forceinline__ const T* bwd_skip_plane(const T* __restrict__ gout, const Dims& d, unsigned row, int* r) {
  const unsigned plane = row / (unsigned)d.H2;
  *r = (int)(row - plane * (unsigned)d.H2);
  const unsigned b = plane / (unsigned)d.Cs;
  const unsigned ch = plane - b * (unsigned)d.Cs;
  return gout + (size_t)(b * (unsigned)d.C + (unsigned)d.Cx + ch) * ((size_t)d.Ho * d.Wo);
}

// grad_x (B,Cx,h,w) in chunks [0, chunks_x), then grad_skip (B,Cs,H2,W2) in chunks [chunks_x, chunks_x + chunks_s)
template <typename T>
__global__ void __launch_bounds__(kT) k_upcat_pad_bwd(const T* __restrict__ gout, T* __restrict__ gx,
                                                      T* __restrict__ gskip, Dims d, unsigned nx, unsigned ns,
                                                      unsigned chunks_x, bool aligned_x, bool aligned_s) {
  constexpr int V = Chunk<T>::V;
  const unsigned chunk = blockIdx.x * (unsigned)blockDim.x + threadIdx.x;
  const bool is_x = chunk < chunks_x;
  const unsigned e0 = (is_x ? chunk : chunk - chunks_x) * (unsigned)V;
  const unsigned n = is_x ? nx : ns;
  if (e0 >= n) return;
  const int cnt = n - e0 < (unsigned)V ? (int)(n - e0) : V;
  Chunk<T> c;
  if (is_x) {
    const int up = 1 << d.up_shift;
    unsigned row = e0 / (unsigned)d.w;
    int j = (int)(e0 - row * (unsigned)d.w);
    int i;
    const T* g = bwd_x_plane(gout, d, row, &i);
#pragma unroll
    for (int k = 0; k < V; ++k) {
      if (k < cnt) {
        if (j == d.w) {
          j = 0;
          g = bwd_x_plane(gout, d, ++row, &i);
        }
        // children row-major, as ATen sums them from 0.0f (a fold is never -0.0f, so 0.0f + fold == fold)
        float acc = fold(g, up * i, up * j, d);
        if (up == 2) {
          acc += fold(g, 2 * i, 2 * j + 1, d);
          acc += fold(g, 2 * i + 1, 2 * j, d);
          acc += fold(g, 2 * i + 1, 2 * j + 1, d);
        }
        c.v[k] = fromf<T>(acc);
        ++j;
      }
    }
    store_chunk(gx + e0, c, cnt, aligned_x);
  } else {
    unsigned row = e0 / (unsigned)d.W2;
    int q = (int)(e0 - row * (unsigned)d.W2);
    int r;
    const T* g = bwd_skip_plane(gout, d, row, &r);
#pragma unroll
    for (int k = 0; k < V; ++k) {
      if (k < cnt) {
        if (q == d.W2) {
          q = 0;
          g = bwd_skip_plane(gout, d, ++row, &r);
        }
        c.v[k] = fromf<T>(fold(g, r, q, d));
        ++q;
      }
    }
    store_chunk(gskip + e0, c, cnt, aligned_s);
  }
}

// -------------------------------------------------------------------------------------------------- host side
int rc(cudaError_t e) { return e == cudaSuccess ? MD2_OK : MD2_ERR_CUDA; }

size_t dtype_size(int dtype) { return dtype == MD2_DTYPE_F32 ? 4 : 2; }

bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

// argument checks shared by both directions; fills d and the element counts (which must fit 32-bit indices)
int make_dims(int dtype, int batch, int x_channels, int skip_channels, int height, int width, int up, Dims* d,
              unsigned* n_out, unsigned* n_x, unsigned* n_skip) {
  if (dtype != MD2_DTYPE_F32 && dtype != MD2_DTYPE_BF16 && dtype != MD2_DTYPE_F16) return MD2_ERR_INVALID_ARGUMENT;
  if (up != 1 && up != 2) return MD2_ERR_INVALID_ARGUMENT;
  if (batch < 1 || x_channels < 1 || skip_channels < 0 || height < 1 || width < 1) return MD2_ERR_INVALID_ARGUMENT;
  const long long H2 = (long long)up * height, W2 = (long long)up * width;
  if (H2 < 2 || W2 < 2) return MD2_ERR_INVALID_ARGUMENT;               // ReflectionPad2d(1) needs 2 values an axis
  const long long C = (long long)x_channels + skip_channels;
  const long long out = (long long)batch * C * (H2 + 2) * (W2 + 2);
  if (out > INT_MAX) return MD2_ERR_UNSUPPORTED;                        // 32-bit element indices
  d->Cx = x_channels;
  d->Cs = skip_channels;
  d->C = (int)C;
  d->h = height;
  d->w = width;
  d->H2 = (int)H2;
  d->W2 = (int)W2;
  d->Ho = (int)H2 + 2;
  d->Wo = (int)W2 + 2;
  d->up_shift = up == 2 ? 1 : 0;
  *n_out = (unsigned)out;
  *n_x = (unsigned)((long long)batch * x_channels * height * width);
  *n_skip = (unsigned)((long long)batch * skip_channels * H2 * W2);
  return MD2_OK;
}

template <typename T>
int launch_fwd(const void* x, const void* skip, void* out, const Dims& d, unsigned n, cudaStream_t s) {
  constexpr unsigned V = Chunk<T>::V;
  const unsigned chunks = (n + V - 1) / V;
  k_upcat_pad<T><<<(chunks + kT - 1) / kT, kT, 0, s>>>((const T*)x, (const T*)skip, (T*)out, d, n, aligned16(out));
  return rc(cudaGetLastError());
}

template <typename T>
int launch_bwd(const void* gout, void* gx, void* gskip, const Dims& d, unsigned nx, unsigned ns, cudaStream_t s) {
  constexpr unsigned V = Chunk<T>::V;
  const unsigned cx = (nx + V - 1) / V, cs = (ns + V - 1) / V;
  const unsigned chunks = cx + cs;
  if (chunks == 0) return MD2_OK;
  k_upcat_pad_bwd<T><<<(chunks + kT - 1) / kT, kT, 0, s>>>((const T*)gout, (T*)gx, (T*)gskip, d, nx, ns, cx,
                                                            aligned16(gx), aligned16(gskip));
  return rc(cudaGetLastError());
}

}  // namespace

extern "C" {

int md2_upcat_pad(const void* x, const void* skip, void* out, int dtype, int batch, int x_channels, int skip_channels,
                  int height, int width, int up, void* stream) {
  Dims d;
  unsigned n, nx, ns;
  const int st = make_dims(dtype, batch, x_channels, skip_channels, height, width, up, &d, &n, &nx, &ns);
  if (st != MD2_OK) return st;
  if (!x || !out || (skip_channels > 0 && !skip)) return MD2_ERR_INVALID_ARGUMENT;
  const cudaStream_t s = (cudaStream_t)stream;
  switch (dtype) {
    case MD2_DTYPE_F32: return launch_fwd<float>(x, skip, out, d, n, s);
    case MD2_DTYPE_BF16: return launch_fwd<__nv_bfloat16>(x, skip, out, d, n, s);
    default: return launch_fwd<__half>(x, skip, out, d, n, s);
  }
}

int md2_upcat_pad_backward(const void* grad_out, void* grad_x, void* grad_skip, int dtype, int batch, int x_channels,
                           int skip_channels, int height, int width, int up, void* stream) {
  Dims d;
  unsigned n, nx, ns;
  const int st = make_dims(dtype, batch, x_channels, skip_channels, height, width, up, &d, &n, &nx, &ns);
  if (st != MD2_OK) return st;
  if (!grad_out) return MD2_ERR_INVALID_ARGUMENT;
  if (!grad_x) nx = 0;
  if (!grad_skip) ns = 0;
  const cudaStream_t s = (cudaStream_t)stream;
  switch (dtype) {
    case MD2_DTYPE_F32: return launch_bwd<float>(grad_out, grad_x, grad_skip, d, nx, ns, s);
    case MD2_DTYPE_BF16: return launch_bwd<__nv_bfloat16>(grad_out, grad_x, grad_skip, d, nx, ns, s);
    default: return launch_bwd<__half>(grad_out, grad_x, grad_skip, d, nx, ns, s);
  }
}

}  // extern "C"
