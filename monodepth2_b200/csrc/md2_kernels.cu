// md2_kernels.cu - sm_100a kernels of the fused view-synthesis loss and their launcher.
//
// Launch sequence of one md2_view_synthesis_loss() call (one stream, no host sync):
//   1. md2_prologue        zero the accumulators, build the per-(sample,source) projection
//  1b. md2_pack            target / sources NCHW -> RGBx texels (B,H,W,4)
//   2. md2_disp_mean       per-sample mean of disp_s            (trainer.py:486)
//   3. md2_identity        scale-independent identity losses    (trainer.py:432-439)
//   4. md2_smooth          edge-aware smoothness, fwd + numerator gradient (layers.py:202-215)
//   5. md2_march_roles     fused warp + photometric loss + min/automask + adjoint, all scales
//   6. md2_final           up-sampling adjoint + smoothness adjoint -> grad_disp_s, losses, grad_T
//
// md2_march_roles (md2_roles.cuh) is the hot kernel.  One CTA owns a band of 28 columns and marches
// down a segment of rows; lane l of each warp holds column x0-2+l, and the warps of the CTA split the
// stages of a row between them (see md2_roles.cuh).  No tensor cores (the path is gather/stream work,
// BASELINE.json).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>

#include <mutex>

#include "md2_core.cuh"
#include "md2_pack2.cuh"
#include "md2_plan.h"

namespace md2 {

constexpr int kWarpsPerCta = 4;          // identity pass (register-marching form): one job per warp
constexpr int kThreads = kWarpsPerCta * 32;
constexpr unsigned kFull = 0xffffffffu;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

}  // namespace md2
#include "md2_roles.cuh"
namespace md2 {

// ------------------------------------------------------------------ 1. prologue
__global__ void md2_prologue(Params P) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const int nacc = acc_count(P);
  for (int i = tid; i < nacc; i += gridDim.x * blockDim.x) P.acc[i] = 0.0;
  // (posecnn: the projections depend on the mean inverse depth of every scale and are built by md2_posecnn_setup)
  if (!P.posecnn)
    for (int i = tid; i < P.B * P.nsrc; i += gridDim.x * blockDim.x) setup_projection(P, 0, i / P.nsrc, i % P.nsrc);
}

// ------------------------------------------------------------------ posecnn (trainer.py:366-375)
// sum of the up-sampled disparity of every (scale, sample) over the full-resolution grid: one thread per fine pixel
__global__ void __launch_bounds__(256) md2_updisp_sum(Params P) {
  const int s = blockIdx.z, b = blockIdx.y;
  const int lv = P.lvl[s], Hs = P.H >> lv, Ws = P.W >> lv, n = P.H * P.W;
  const float* d = P.disp[s] + (size_t)b * Hs * Ws;
  float a = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    a += upsample_at(d, lv, Hs, Ws, i / P.W, i % P.W);
  a = warp_sum(a);
  __shared__ float part[8];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) part[w] = a;
  __syncthreads();
  if (w == 0) {
    a = (l < 8) ? part[l] : 0.f;
    a = warp_sum(a);
    if (l == 0) atomicAdd(&P.acc[acc_updisp(P, s, b)], (double)a);
  }
}
// mean inverse depth, then T and the projection table of every (scale, sample, source)
__global__ void md2_posecnn_setup(Params P) {
  const int b = blockIdx.x, s = threadIdx.x;
  if (s < P.S) posecnn_mid(P, s, b);
  __syncthreads();
  for (int i = threadIdx.x; i < P.S * P.nsrc; i += blockDim.x) setup_projection(P, i / P.nsrc, b, i % P.nsrc);
}
// pose epilogue of every sample (gradients of the leaves, and the constant each scale adds to d loss / d up-sampled
// disparity), then that constant for scale 0, whose gradient the marching pass has already finished
__global__ void md2_posecnn_final(Params P) {
  const int b = blockIdx.x;
  if (threadIdx.x == 0) final_pose_posecnn(P, b);
  __syncthreads();
  if (P.up0 == 0) return;        // no level-0 slot: every level adds its constant in the up-sampling adjoint
  const float cst = P.gmidc[b];
  float* g = P.grad_disp[0] + (size_t)b * P.H * P.W;
  for (int i = threadIdx.x; i < P.H * P.W; i += blockDim.x) g[i] += cst;
}

// ------------------------------------------------------------------ --predictive_mask (trainer.py:447-459)
// masks up-sampled to full resolution (read by the marching pass) + the BCE sums
__global__ void __launch_bounds__(256) md2_pmask_up(Params P) {
  const int s = blockIdx.z, bf = blockIdx.y;
  const int n = P.H * P.W;
  float a = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    a += pmask_up_pixel(P, s, bf / P.nsrc, bf % P.nsrc, i / P.W, i % P.W);
  a = warp_sum(a);
  __shared__ float part[8];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) part[w] = a;
  __syncthreads();
  if (w == 0) {
    a = (l < 8) ? part[l] : 0.f;
    a = warp_sum(a);
    if (l == 0) atomicAdd(&P.acc[acc_bce(P, s)], (double)a);
  }
}
// d loss / d mask_s: adjoint of the up-sampling over (photometric part + BCE part), one thread per coarse pixel
__global__ void __launch_bounds__(256) md2_pmask_grad(Params P) {
  const int s = blockIdx.z, bf = blockIdx.y;
  if (!P.grad_pmask[s]) return;
  const int Hs = P.H >> P.lvl[s], Ws = P.W >> P.lvl[s];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < Hs * Ws) pmask_grad_pixel(P, s, bf / P.nsrc, bf % P.nsrc, i / Ws, i % Ws);
}

// re-layout of target and sources to RGBx texels (one 16-byte load per bilinear tap later on)
__global__ void md2_pack(Params P) {
  const int img = blockIdx.z, b = blockIdx.y;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < P.H * P.W) pack_pixel(P, img, b, p);
}

// ------------------------------------------------------------------ 2. disparity means
__global__ void md2_disp_mean(Params P) {
  const int s = blockIdx.z, b = blockIdx.y;
  if (s >= P.S) return;
  const int n = (P.H >> P.lvl[s]) * (P.W >> P.lvl[s]);
  if (blockIdx.x * blockDim.x >= n) return;                      // uniform per block
  const float* d = P.disp[s] + (size_t)b * n;
  float a = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) a += __ldg(d + i);
  a = warp_sum(a);
  __shared__ float part[32];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) part[w] = a;
  __syncthreads();
  if (w == 0) {
    a = (l < (blockDim.x >> 5)) ? part[l] : 0.f;
    a = warp_sum(a);
    if (l == 0) atomicAdd(&P.acc[acc_dispsum(P, s, b)], (double)a);
  }
}

// ------------------------------------------------------------------ 2b. depth planes of the up-sampled disparities
// zup[s](b, y, x) = disp_to_depth(bilinear_up(disp_s)(y, x))    (trainer.py:349-353, layers.py:16-25): what role A of the
// role-specialised marching kernel used to rebuild per row and lane from four disparity taps.  The expressions are the
// ones of prefetch_row / lane_init / stage_a_issue (md2_core.cuh), term by term, so the values are the same.
constexpr int kDupCols = 128, kDupRows = 16;                  // fine pixels per block of md2_depth_up
__global__ void __launch_bounds__(256) md2_depth_up(Params P) {
  // block = 256 threads, tile = 128 columns x 16 rows of the full-resolution plane; blockIdx.z = b * (S - up0) + s - up0,
  // slots s >= up0, i.e. levels >= 1 (level 0 is not up-sampled: its readers take the disparity plane and apply disp_to_depth themselves).
  // Separable, through shared memory: pass 1 blends every coarse row the tile touches horizontally (top / bot of
  // stage_a_issue: the same up_blend on the same operands), pass 2 blends two of those rows vertically and applies
  // disp_to_depth - the x weights are computed once per column of the tile instead of once per pixel.
  __shared__ __align__(16) float hrow[kDupRows / 2 + 2][kDupCols];
  const int nup = P.S - P.up0;
  const int s = P.up0 + blockIdx.z % nup, b = blockIdx.z / nup;
  const int Hs = P.H >> P.lvl[s], Ws = P.W >> P.lvl[s];
  const float rs = 1.0f / (float)(1 << P.lvl[s]);
  const float* d = P.disp[s] + (size_t)b * Hs * Ws;
  const int x_base = blockIdx.x * kDupCols, y_base = blockIdx.y * kDupRows;
  // coarse rows touched by fine rows [y_base, y_base + kDupRows): y0 of the first row .. y1 of the last row
  auto src_row = [&](int y, int& y0, int& y1, float& l1) {
    float syr = fmaf(rs, (float)y + 0.5f, -0.5f);
    syr = syr < 0.0f ? 0.0f : syr;
    y0 = (int)syr;
    y1 = y0 + ((y0 < Hs - 1) ? 1 : 0);
    l1 = syr - (float)(int)syr;
  };
  int cy_lo, cy_tmp, cy_hi;
  float ltmp;
  src_row(y_base, cy_lo, cy_tmp, ltmp);
  src_row(min(y_base + kDupRows, P.H) - 1, cy_tmp, cy_hi, ltmp);
  const int ncy = cy_hi - cy_lo + 1;                          // <= kDupRows / 2 + 2 for s >= 1
  // pass 1: thread -> (coarse row, fine column)
  for (int i = threadIdx.x; i < ncy * kDupCols; i += 256) {
    const int r = i / kDupCols, cx = i - r * kDupCols;
    const int x = min(x_base + cx, P.W - 1);
    float sxr = fmaf(rs, (float)x + 0.5f, -0.5f);
    sxr = sxr < 0.0f ? 0.0f : sxr;
    const int ux0 = (int)sxr;
    const int ux1 = ux0 + ((ux0 < Ws - 1) ? 1 : 0);
    const float ul1 = sxr - (float)ux0;
    const float ul0 = 1.0f - ul1;
    const float* row = d + (cy_lo + r) * Ws;
    hrow[r][cx] = up_blend(ul0, __ldg(row + ux0), ul1, __ldg(row + ux1));
  }
  __syncthreads();
  // pass 2: thread -> 4 consecutive columns of 2 rows (32 threads x 4 columns = 128 columns, 8 thread rows x 2)
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int x4 = x_base + tx * 4;
  if (x4 >= P.W) return;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int y = y_base + ty * 2 + k;
    if (y >= P.H) break;
    int y0, y1;
    float l1;
    src_row(y, y0, y1, l1);
    const float l0 = 1.0f - l1;
    const float4 a4 = *reinterpret_cast<const float4*>(hrow[y0 - cy_lo] + tx * 4);
    const float4 b4 = *reinterpret_cast<const float4*>(hrow[y1 - cy_lo] + tx * 4);
    const float h0[4] = {a4.x, a4.y, a4.z, a4.w}, h1[4] = {b4.x, b4.y, b4.z, b4.w};
    float z[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) z[i] = depth_of_disp(P, up_blend(l0, h0[i], l1, h1[i]));
    float* out = P.zup[s] + (size_t)b * P.H * P.W + y * P.W + x4;
    if ((P.W & 3) == 0) {
      *reinterpret_cast<float4*>(out) = make_float4(z[0], z[1], z[2], z[3]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (x4 + i < P.W) out[i] = z[i];
    }
  }
}

// ------------------------------------------------------------------ 3. identity losses
template <int NSRC, bool NOSSIM>
__global__ void __launch_bounds__(kThreads) md2_identity(Params P) {
  const int lane = threadIdx.x & 31;
  const int job = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  const int njobs = P.B * P.nseg_id * P.nband_id;
  if (job >= njobs) return;
  const int band = job % P.nband_id;
  const int seg = (job / P.nband_id) % P.nseg_id;
  const int b = job / (P.nband_id * P.nseg_id);
  const int y0 = seg * P.id_rows;
  const int y1 = min(y0 + P.id_rows, P.H);
  IdLane<NSRC> L;
  id_init(L, P, band * kIdCols, lane);
  id_prefetch(L, P, b, y0 - 1);
  for (int t = y0 - 1; t <= y1; ++t) {
    id_stage_a(L, P, b, t, lane, y0, y1);
    IdXchg<NSRC> lf, rt;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      lf.tg[c] = __shfl_up_sync(kFull, L.tg[c], 1);
      rt.tg[c] = __shfl_down_sync(kFull, L.tg[c], 1);
#pragma unroll
      for (int f = 0; f < NSRC; ++f) {
        lf.pr[f][c] = __shfl_up_sync(kFull, L.pr[f][c], 1);
        rt.pr[f][c] = __shfl_down_sync(kFull, L.pr[f][c], 1);
      }
    }
    id_stage_b<NSRC, NOSSIM>(L, P, b, t, lane, y0, y1, lf, rt);
  }
}

// packed-fp32 form of the identity pass for two sources (md2_pack2.cuh)
template <bool NOSSIM>
__global__ void __launch_bounds__(kThreads) md2_identity2(Params P) {
  const int lane = threadIdx.x & 31;
  const int job = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  const int njobs = P.B * P.nseg_id * P.nband_id;
  if (job >= njobs) return;
  const int band = job % P.nband_id;
  const int seg = (job / P.nband_id) % P.nseg_id;
  const int b = job / (P.nband_id * P.nseg_id);
  const int y0 = seg * P.id_rows;
  const int y1 = min(y0 + P.id_rows, P.H);
  IdLane2 L;
  id_init2(L, P, band * kIdCols, lane);
  id_prefetch2(L, P, b, y0 - 1);
  id_shift2(L);
  id_prefetch2(L, P, b, y0);
  for (int t = y0 - 1; t <= y1; ++t) {
    id_stage_a2(L, P, b, t, lane, y0, y1);
    IdXchg2 lf, rt;
    lf.tgrg = p2(__shfl_up_sync(kFull, L.tgrg.x, 1), __shfl_up_sync(kFull, L.tgrg.y, 1));
    rt.tgrg = p2(__shfl_down_sync(kFull, L.tgrg.x, 1), __shfl_down_sync(kFull, L.tgrg.y, 1));
    lf.tgb = __shfl_up_sync(kFull, L.tgb, 1);
    rt.tgb = __shfl_down_sync(kFull, L.tgb, 1);
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      lf.pr[s] = p2(__shfl_up_sync(kFull, L.pr[s].x, 1), __shfl_up_sync(kFull, L.pr[s].y, 1));
      rt.pr[s] = p2(__shfl_down_sync(kFull, L.pr[s].x, 1), __shfl_down_sync(kFull, L.pr[s].y, 1));
    }
    id_stage_b2<NOSSIM>(L, P, b, t, lane, y0, y1, lf, rt);
  }
}

// ------------------------------------------------------------------ 3b. identity pass, TMA-staged
// The identity pass is a streaming stencil: every input byte is used by a 3x3 window and nothing is
// data-dependent, so the tile a CTA needs is a box.  One elected thread arms an mbarrier and issues three
// cp.async.bulk.tensor (TMA) loads - target, source 0, source 1, each a box of kTmaBoxW x kTmaBoxH x 3 channels of
// the planar (B*3, H, W) tensor including the 1-pixel halo - the CTA waits on the barrier, mirrors the halo of
// border tiles in shared memory (TMA fills out-of-bounds elements with zeros, ReflectionPad2d(1) wants the
// mirror image, layers.py:235-236) and marches the rows out of shared memory: a lane owns one column and reads
// its left / right neighbours from the tile (no warp halo, no shuffles, all 32 lanes productive).  Four CTAs per
// SM (4 x 48 KB of tiles) overlap the loads of some CTAs with the arithmetic of the others.  Used for two sources when the
// row pitch is a multiple of 16 bytes; otherwise md2_identity / md2_identity2 run.
// kTmaRows measured (whole step, 640x192 x 12): 8 rows 0.486 ms, 12 rows 0.487 ms, 16 rows 0.491 ms
constexpr int kTmaCols = 128, kTmaRows = 8;                   // pixels a CTA owns
constexpr int kTmaPadX = 4;      // the box starts 4 columns left of the tile: TMA needs a 16-byte aligned inner start
constexpr int kTmaBoxW = kTmaCols + 2 * kTmaPadX, kTmaBoxH = kTmaRows + 2;   // (x0 - 1 faults with "illegal instruction")
constexpr int kTmaImgFloats = ((3 * kTmaBoxH * kTmaBoxW * 4 + 127) / 128) * 32;   // one image's tile, 128-byte multiple
constexpr int tma_smem_bytes(int nsrc) { return (1 + nsrc) * kTmaImgFloats * 4 + 16; }

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

struct IdTensorMaps { CUtensorMap img[1 + kMaxSrc]; };     // target, then the sources

template <int NSRC, bool NOSSIM>
__global__ void __launch_bounds__(kTmaCols) md2_identity_tma(Params P, const __grid_constant__ IdTensorMaps maps) {
  constexpr int NIMG = 1 + NSRC;
  extern __shared__ __align__(128) float tile[];
  unsigned long long* bar = reinterpret_cast<unsigned long long*>(tile + NIMG * kTmaImgFloats);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int x0 = blockIdx.x * kTmaCols, y0 = blockIdx.y * kTmaRows, b = blockIdx.z;
  const int y1 = min(y0 + kTmaRows, P.H);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned bytes = (unsigned)NIMG * 3u * kTmaBoxH * kTmaBoxW * 4u;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
#pragma unroll
    for (int i = 0; i < NIMG; ++i)
      asm volatile(
          "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
          ::"r"(smem_u32(tile + i * kTmaImgFloats)), "l"(&maps.img[i]), "r"(x0 - kTmaPadX), "r"(y0 - 1), "r"(b * 3),
            "r"(smem_u32(bar))
          : "memory");
  }
  {   // every thread waits for the bytes to land (phase 0)
    unsigned done = 0, spins = 0;
    while (!done) {
      asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
                   : "=r"(done) : "r"(smem_u32(bar)) : "memory");
#if defined(MD2_BOUNDS_CHECK)
      // debug build only: a tensor-map fault must not turn into a hang of the test run.  The product build waits
      // (a slow but valid completion - time slicing, MPS, a profiler replay - must not kill the CUDA context).
      if (!done && ++spins > (1u << 26)) __trap();
#else
      (void)spins;
#endif
    }
  }
  __syncthreads();                  // every thread has observed phase 0: the barrier is not used again
  if (threadIdx.x == 0) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
  // mirror the halo of border tiles: columns first, then rows (so that the corners come out right)
  auto at = [&](int img, int c, int r, int col) -> float& { return tile[img * kTmaImgFloats + (c * kTmaBoxH + r) * kTmaBoxW + col]; };
  const int cl = (x0 == 0) ? kTmaPadX - 1 : -1;                           // tile column of x = -1
  const int cr = (P.W - x0 + kTmaPadX <= kTmaBoxW - 1) ? P.W - x0 + kTmaPadX : -1;   // tile column of x = W
  if (cl >= 0 || cr >= 0) {
    for (int i = threadIdx.x; i < NIMG * 3 * kTmaBoxH; i += blockDim.x) {
      const int img = i / (3 * kTmaBoxH), c = (i / kTmaBoxH) % 3, r = i % kTmaBoxH;
      if (cl >= 0) at(img, c, r, cl) = at(img, c, r, cl + 2);
      if (cr >= 2) at(img, c, r, cr) = at(img, c, r, cr - 2);
    }
    __syncthreads();
  }
  const int rt_ = (y0 == 0) ? 0 : -1;                                     // tile row of y = -1
  const int rb = (P.H - y0 + 1 <= kTmaBoxH - 1 && P.H >= y0) ? P.H - y0 + 1 : -1;   // tile row of y = H
  if (rt_ >= 0 || rb >= 0) {
    for (int i = threadIdx.x; i < NIMG * 3 * kTmaBoxW; i += blockDim.x) {
      const int img = i / (3 * kTmaBoxW), c = (i / kTmaBoxW) % 3, col = i % kTmaBoxW;
      if (rt_ >= 0) at(img, c, 0, col) = at(img, c, 2, col);
      if (rb >= 2) at(img, c, rb, col) = at(img, c, rb - 2, col);
    }
    __syncthreads();
  }
  const int x = x0 + warp * 32 + lane;
  const bool colok = x < P.W;
  const int col = warp * 32 + lane + kTmaPadX;                            // tile column of this lane's pixel
  const int plane = P.H * P.W;
  // NSRC == 2: packed-fp32 arithmetic (md2_pack2.cuh); otherwise the scalar stage of md2_core.cuh
  IdLane2 L2;
  IdLane<NSRC> L1;
  if constexpr (NSRC == 2) { id_init2(L2, P, 0, 0); L2.x = x; L2.colok = colok; L2.xi = colok ? x : P.W - 1; }
  else { id_init(L1, P, 0, 0); L1.x = x; L1.colok = colok; L1.xi = colok ? x : P.W - 1; }
  for (int r = 0; r < kTmaBoxH; ++r) {
    const int t = y0 - 1 + r;
    if (t > y1) break;
    float v[NIMG][3][3];                                                  // [image][channel][left, centre, right]
#pragma unroll
    for (int img = 0; img < NIMG; ++img)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float* row = &at(img, c, r, col);
        v[img][c][0] = row[-1]; v[img][c][1] = row[0]; v[img][c][2] = row[1];
      }
    if (colok && t >= y0 && t < y1) {                                     // RGBx texels for the marching kernel
      const int o4 = 4 * (b * plane + t * P.W + x);
      *reinterpret_cast<float4*>(P.tgt4 + o4) = make_float4(v[0][0][1], v[0][1][1], v[0][2][1], 0.f);
#pragma unroll
      for (int f = 0; f < NSRC; ++f)
        *reinterpret_cast<float4*>(P.src4[f] + o4) = make_float4(v[1 + f][0][1], v[1 + f][1][1], v[1 + f][2][1], 0.f);
    }
    if constexpr (NSRC == 2) {
      IdXchg2 lf, rt;
      lf.tgrg = p2(v[0][0][0], v[0][1][0]); lf.tgb = v[0][2][0];
      rt.tgrg = p2(v[0][0][2], v[0][1][2]); rt.tgb = v[0][2][2];
      L2.tgrg = p2(v[0][0][1], v[0][1][1]); L2.tgb = v[0][2][1];
      lf.pr[0] = p2(v[1][0][0], v[1][1][0]); lf.pr[1] = p2(v[2][0][0], v[2][1][0]); lf.pr[2] = p2(v[1][2][0], v[2][2][0]);
      rt.pr[0] = p2(v[1][0][2], v[1][1][2]); rt.pr[1] = p2(v[2][0][2], v[2][1][2]); rt.pr[2] = p2(v[1][2][2], v[2][2][2]);
      L2.pr[0] = p2(v[1][0][1], v[1][1][1]); L2.pr[1] = p2(v[2][0][1], v[2][1][1]); L2.pr[2] = p2(v[1][2][1], v[2][2][1]);
      id_stage_b2<NOSSIM>(L2, P, b, t, lane, y0, y1, lf, rt, 0, 31);
    } else {
      IdXchg<NSRC> lf, rt;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        lf.tg[c] = v[0][c][0]; L1.tg[c] = v[0][c][1]; rt.tg[c] = v[0][c][2];
#pragma unroll
        for (int f = 0; f < NSRC; ++f) { lf.pr[f][c] = v[1 + f][c][0]; L1.pr[f][c] = v[1 + f][c][1]; rt.pr[f][c] = v[1 + f][c][2]; }
      }
      id_stage_b<NSRC, NOSSIM>(L1, P, b, t, lane, y0, y1, lf, rt, 0, 31);
    }
  }
}

// host: tensor map of a planar (B*3, H, W) fp32 image tensor with the identity pass's box
typedef CUresult (*md2_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static md2_encode_tiled_fn get_encode_tiled() {
  static md2_encode_tiled_fn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (md2_encode_tiled_fn)p;
  }();
  return fn;
}
static bool make_image_map(CUtensorMap* m, const float* base, int B, int H, int W) {
  md2_encode_tiled_fn enc = get_encode_tiled();
  if (!enc) return false;
  const cuuint64_t gdim[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B * 3};
  const cuuint64_t gstride[2] = {(cuuint64_t)W * 4, (cuuint64_t)H * W * 4};
  const cuuint32_t box[3] = {kTmaBoxW, kTmaBoxH, 3};
  const cuuint32_t estr[3] = {1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), gdim, gstride, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// ------------------------------------------------------------------ 4. smoothness
// Edge-aware smoothness (layers.py:202-215 on the mean-normalised disparity, trainer.py:486-487): value and
// numerator gradient gn, all scales.  A warp owns 32 columns x kSmoothRows rows of one (scale, sample) and marches
// down: the current row lives in registers, the next row is loaded once, so every edge is evaluated ONCE (its
// weight exp(-|dI|) and sign serve both of its end points: right neighbour by shuffle, upper neighbour from
// the previous step) instead of once per end point.  Same per-edge arithmetic as smooth_pixel (md2_core.cuh).
constexpr int kSmoothRows = 16;
constexpr int kSmoothWarps = 4;
__host__ __device__ inline int smooth_bands(int Ws) { return (Ws + 31) / 32; }
__host__ __device__ inline int smooth_segs(int Hs) { return (Hs + kSmoothRows - 1) / kSmoothRows; }

struct SmoothPx { float raw, n, i0, i1, i2; };
// the colour image of one (scale, sample): float planar, or uint8 planar / interleaved (Params::color8)
struct SmoothImg { const float* f32; const unsigned char* u8; int hwc; };
__device__ __forceinline__ SmoothPx smooth_load(const float* d, const SmoothImg& im, int plane, int p, float inv_m) {
  SmoothPx r;
  r.raw = __ldg(d + p);
  r.n = r.raw * inv_m;
  if (im.u8) {
    const unsigned char* q = im.u8 + (im.hwc ? 3 * p : p);
    const int cs = im.hwc ? 1 : plane;
    r.i0 = u8_unit(__ldg(q)); r.i1 = u8_unit(__ldg(q + cs)); r.i2 = u8_unit(__ldg(q + 2 * cs));
  } else {
    r.i0 = __ldg(im.f32 + p); r.i1 = __ldg(im.f32 + plane + p); r.i2 = __ldg(im.f32 + 2 * plane + p);
  }
  return r;
}
// edge between `a` (first end) and `q`: |n_a - n_q| w  and  sign(n_a - n_q) w
__device__ __forceinline__ void smooth_edge(const SmoothPx& a, const SmoothPx& q, float& e, float& sw) {
  const float g = fabsf(a.i0 - q.i0) + fabsf(a.i1 - q.i1) + fabsf(a.i2 - q.i2);
  const float w = md2_exp_neg(g * (1.0f / 3.0f));
  const float df = a.n - q.n;
  e = fabsf(df) * w;
  sw = (df > 0.f) ? w : ((df < 0.f) ? -w : 0.f);
}

__global__ void __launch_bounds__(kSmoothWarps * 32) md2_smooth(Params P) {
  const int lane = threadIdx.x & 31;
  int rem = blockIdx.x * kSmoothWarps + (threadIdx.x >> 5);
  int s = 0;
  for (; s < P.S; ++s) {
    const int n = smooth_bands(P.W >> P.lvl[s]) * smooth_segs(P.H >> P.lvl[s]) * P.B;
    if (rem < n) break;
    rem -= n;
  }
  if (s >= P.S) return;
  const int Hs = P.H >> P.lvl[s], Ws = P.W >> P.lvl[s], plane = Hs * Ws;
  const int nb = smooth_bands(Ws), ns = smooth_segs(Hs);
  const int b = rem / (nb * ns);
  const int r = rem - b * nb * ns;
  const int seg = r / nb, band = r - seg * nb;
  float inv_m = 0.f;
  if (lane == 0) inv_m = 1.0f / ((float)(P.acc[acc_dispsum(P, s, b)] / (double)plane) + 1e-7f);
  inv_m = __shfl_sync(kFull, inv_m, 0);
  const float* d = P.disp[s] + (size_t)b * plane;
  SmoothImg im;
  im.f32 = P.color[s] ? P.color[s] + (size_t)b * 3 * plane : nullptr;
  im.u8 = P.color8[s] ? P.color8[s] + (size_t)b * 3 * plane : nullptr;
  im.hwc = P.u8_hwc;
  float* gn = P.gn[s] + (size_t)b * plane;
  const float inx = 1.0f / ((float)P.B * (float)Hs * (float)(Ws - 1));
  const float iny = 1.0f / ((float)P.B * (float)(Hs - 1) * (float)Ws);
  const int x = band * 32 + lane;
  const bool xok = x < Ws;
  const int xc = xok ? x : Ws - 1;
  const bool has_rt = x + 1 < Ws;
  // pixel beyond the band that only the first / last lane needs: the left neighbour of lane 0, the right
  // neighbour of lane 31 (loaded one row ahead like the band itself)
  const bool side_lane = (lane == 0 && x > 0) || (lane == 31 && has_rt);
  const int xs = (lane == 0) ? x - 1 : x + 1;
  const int y0 = seg * kSmoothRows, y1 = min(y0 + kSmoothRows, Hs);
  auto row = [&](int y) { return (y < Hs ? y : Hs - 1) * Ws; };
  SmoothPx cur = smooth_load(d, im, plane, row(y0) + xc, inv_m);
  SmoothPx nxt = smooth_load(d, im, plane, row(y0 + 1) + xc, inv_m);
  SmoothPx side = cur, side_nxt = cur;
  if (side_lane) { side = smooth_load(d, im, plane, row(y0) + xs, inv_m); side_nxt = smooth_load(d, im, plane, row(y0 + 1) + xs, inv_m); }
  float sy_up = 0.f;                       // sign * weight of the edge to the row above
  if (y0 > 0) {
    const SmoothPx up = smooth_load(d, im, plane, (y0 - 1) * Ws + xc, inv_m);
    float e;
    smooth_edge(up, cur, e, sy_up);
  }
  float ex = 0.f, ey = 0.f, dot = 0.f;
  for (int y = y0; y < y1; ++y) {
    // rows y and y+1 are in registers; put row y+2 in flight
    const SmoothPx nn = smooth_load(d, im, plane, row(y + 2) + xc, inv_m);
    SmoothPx side_nn = side_nxt;
    if (side_lane) side_nn = smooth_load(d, im, plane, row(y + 2) + xs, inv_m);
    const bool has_dn = y + 1 < Hs;
    // right neighbour: next lane, or the side pixel at the end of the band
    SmoothPx rt;
    rt.n = __shfl_down_sync(kFull, cur.n, 1); rt.i0 = __shfl_down_sync(kFull, cur.i0, 1);
    rt.i1 = __shfl_down_sync(kFull, cur.i1, 1); rt.i2 = __shfl_down_sync(kFull, cur.i2, 1);
    if (lane == 31) rt = side;
    float e_x = 0.f, sx = 0.f, e_y = 0.f, sy = 0.f;
    if (has_rt) smooth_edge(cur, rt, e_x, sx);
    if (has_dn) smooth_edge(cur, nxt, e_y, sy);
    MD2_DBG(if (xok) {       // signs of the smoothness differences (decision export, debug build only)
      const long o = D.smoff[s] + (long)b * plane + (long)y * Ws + x;
      const float dx = cur.n - rt.n, dy = cur.n - nxt.n;
      if (has_rt) D.smx[o] = (signed char)(dx > 0.f ? 1 : (dx < 0.f ? -1 : 0));
      if (has_dn) D.smy[o] = (signed char)(dy > 0.f ? 1 : (dy < 0.f ? -1 : 0));
    });
    // left neighbour's edge towards this pixel: previous lane, or recomputed from the side pixel
    float sxl = __shfl_up_sync(kFull, sx, 1);
    if (lane == 0) {
      sxl = 0.f;
      if (x > 0) { float e; smooth_edge(side, cur, e, sxl); }
    }
    if (xok) {
      MD2_CHK(y * Ws + x, plane);
      // d(sum_x/Nx + sum_y/Ny) / d n(p): +sign*w for the edges this pixel starts, -sign*w for those it ends
      float g = 0.f;
      g += inx * sx;
      g += inx * (-sxl);
      g += iny * sy;
      g += iny * (-sy_up);
      gn[y * Ws + x] = g;
      ex += e_x; ey += e_y;
      dot = fmaf(g, cur.raw, dot);
    }
    sy_up = sy;
    cur = nxt; nxt = nn;
    side = side_nxt; side_nxt = side_nn;
  }
  ex = warp_sum(ex); ey = warp_sum(ey); dot = warp_sum(dot);
  if (lane == 0) {
    atomicAdd(&P.acc[acc_smx(P, s, b)], (double)ex);
    atomicAdd(&P.acc[acc_smy(P, s, b)], (double)ey);
    atomicAdd(&P.acc[acc_dot(P, s, b)], (double)dot);
  }
}

// per-(scale, sample) scalars of the smoothness adjoint, once, in fp64 (the fp64 pipe is slow on B200:
// doing this at the top of every block of md2_final cost ~20 us)
__global__ void md2_smooth_scalars(Params P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.S * P.B) return;
  float inv_m, dterm;
  smooth_scalars(P, i / P.B, i % P.B, inv_m, dterm);
  P.smsc[2 * i] = inv_m;
  P.smsc[2 * i + 1] = dterm;
}

// ------------------------------------------------------------------ 6. final
// grad_disp_s (s >= 1) = adjoint of the bilinear up-sampling of dD_s (trainer.py:350-351) + smoothness
// adjoint.  Separable, one pass over the fine map: a block owns kFinalFineRows fine rows x 256 fine columns;
// pass 1, one thread per fine column (coalesced rows), folds the rows into the block's coarse rows with the
// vertical weights and leaves them in shared memory; pass 2, one thread per coarse pixel, folds 2K columns
// with the horizontal weights.  Every fine value is read ~1.1x (the gather form read it 4x).  Block 0 also
// writes the losses and grad_T.  Scale 0 is finished by the marching kernel itself.
constexpr int kFinalThreads = 256;
// (measured at 640x192 x 12, 1 296 blocks = 1.09 waves with 16 rows: 24 rows 16.4 us, 32 rows 17.4 us, 8 rows 16.9 us, 16 rows 15.0 us)
constexpr int kFinalFineRows = 16;

__host__ __device__ inline int final_tiles_x(int Ws, int K) { const int t = kFinalThreads / K - 1; return (Ws + t - 1) / t; }
__host__ __device__ inline int final_tiles_y(int Hs, int K) { const int t = kFinalFineRows / K; return (Hs + t - 1) / t; }

template <int K>
__device__ __forceinline__ void final_tile(const Params& P, int s, int b, int tx, int ty) {
  constexpr int TXC = kFinalThreads / K - 1;     // coarse columns per block
  constexpr int TYC = kFinalFineRows / K;        // coarse rows per block
  constexpr int NR = (TYC + 1) * K;              // fine rows read per block
  __shared__ float sm[TYC][kFinalThreads];
  const int Hs = P.H >> P.lvl[s], Ws = P.W >> P.lvl[s];
  const int X0 = tx * TXC, Y0 = ty * TYC;
  const float* dD = P.dD[s] + (size_t)b * P.H * P.W;
  // posecnn: d loss / d (every pixel of the up-sampled disparity) through mean_inv_depth (fine indices outside the
  // image have weight 0, so the constant may be added to every value read)
  const float cst = P.posecnn ? __ldg(P.gmidc + s * P.B + b) : 0.0f;
  {
    const int x = K * X0 - K / 2 + (int)threadIdx.x;
    const int xc = x < 0 ? 0 : (x >= P.W ? P.W - 1 : x);
    const int ylo = K * Y0 - K / 2;
    float acc[TYC];
#pragma unroll
    for (int l = 0; l < TYC; ++l) acc[l] = 0.f;
    float v[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      const int y = ylo + r;
      const int yc = y < 0 ? 0 : (y >= P.H ? P.H - 1 : y);
      v[r] = __ldg(dD + yc * P.W + xc) + cst;
    }
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      // fine row r is tap r - l*K of coarse row l, for the (at most two) rows l with 0 <= r - l*K < 2K
#pragma unroll
      for (int l = 0; l < TYC; ++l) {
        const int i = r - l * K;
        if (i >= 0 && i < 2 * K) acc[l] = fmaf(up_weight<K>(i, Y0 + l, Hs), v[r], acc[l]);
      }
    }
#pragma unroll
    for (int l = 0; l < TYC; ++l) sm[l][threadIdx.x] = acc[l];
  }
  __syncthreads();
  const float inv_m = __ldg(P.smsc + 2 * (s * P.B + b)), dterm = __ldg(P.smsc + 2 * (s * P.B + b) + 1);
  for (int idx = threadIdx.x; idx < TYC * TXC; idx += kFinalThreads) {
    const int l = idx / TXC, lx = idx - l * TXC;
    const int X = X0 + lx, Y = Y0 + l;
    if (X >= Ws || Y >= Hs) continue;
    float a = 0.f;
#pragma unroll
    for (int i = 0; i < 2 * K; ++i) a = fmaf(up_weight<K>(i, X, Ws), sm[l][lx * K + i], a);
    const int cp = Y * Ws + X;
    P.grad_disp[s][(size_t)b * Hs * Ws + cp] = a + final_smooth_grad(P, s, b, cp, inv_m, dterm);
  }
}

__global__ void __launch_bounds__(kFinalThreads) md2_final(Params P) {
  if (blockIdx.x == 0) {
    if (threadIdx.x == 0) final_scalars(P);
    if (P.want_grad)
      for (int i = threadIdx.x; i < P.B * P.nsrc; i += blockDim.x) final_grad_T(P, i / P.nsrc, i % P.nsrc);
  }
  if (!P.want_grad) return;
  // block -> (scale, sample, tile row, tile column), scale-major
  int rem = blockIdx.x;
  for (int s = P.up0; s < P.S; ++s) {
    const int K = 1 << P.lvl[s];
    const int ntx = final_tiles_x(P.W >> P.lvl[s], K), nty = final_tiles_y(P.H >> P.lvl[s], K);
    const int n = ntx * nty * P.B;
    if (rem < n) {
      const int b = rem / (ntx * nty);
      const int t = rem - b * ntx * nty;
      const int ty = t / ntx, tx = t - ty * ntx;
      switch (K) {
        case 2: final_tile<2>(P, s, b, tx, ty); break;
        case 4: final_tile<4>(P, s, b, tx, ty); break;
        default: final_tile<8>(P, s, b, tx, ty); break;
      }
      return;
    }
    rem -= n;
  }
}

// ------------------------------------------------------------------ launcher

// Whether the two-source kernels that have a packed-fp32 form (md2_pack2.cuh) use it: the marching kernel's roles A
// and B, and the identity pass.  MD2_PACK2=off in the environment forces the scalar form for every call (A/B checks,
// tests/test_gpu_parity.py).
static bool pack2_on() {
#ifdef MD2_DBG_DEVICE
  return false;      // the decision export lives in the scalar stage functions
#else
  static const bool on = [] {
    const char* e = getenv("MD2_PACK2");
    return !(e && !strcmp(e, "off"));
  }();
  return on;
#endif
}

static int device_sm_count() {
  static const int n = [] {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v < 1)
      v = 148;
    return v;
  }();
  return n;
}

template <class C0>
static cudaError_t launch_march_roles(const Params& P0, cudaStream_t stream) {
  typedef RoleOf<C0> C;
  typedef RoleCfg<C> RC;
  Params P = P0;
  P.nsm = device_sm_count();
  const int jobs = P.S * P.B * P.nseg * P.nband;
  const size_t smem = (size_t)RC::SMEM_F4 * sizeof(float4);
  if constexpr (C::NSRC == 2 && !C::AVG && (C::AUTOMASK || !C::GRAD)) {
    if (pack2_on()) {                 // packed-fp32 roles unless MD2_PACK2=off (--disable_automasking with
                                      // gradients: the packed form spills 16 bytes under 128 registers, scalar fits)
      static cudaError_t attr2 = cudaFuncSetAttribute(md2_march_roles<C, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (attr2 != cudaSuccess) return attr2;
      md2_march_roles<C, true><<<jobs, RC::THREADS, smem, stream>>>(P);
      return cudaGetLastError();
    }
  }
  static cudaError_t attr = cudaFuncSetAttribute(md2_march_roles<C, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (attr != cudaSuccess) return attr;
  md2_march_roles<C, false><<<jobs, RC::THREADS, smem, stream>>>(P);
  return cudaGetLastError();
}

template <int NSRC, bool NOSSIM>
static cudaError_t launch_march_n(const Params& P, cudaStream_t stream) {
  const int key = (P.avg ? 4 : 0) | (P.automask ? 2 : 0) | (P.want_grad ? 1 : 0);
  switch (key) {
    case 0: return launch_march_roles<Cfg<NSRC, false, false, false, NOSSIM>>(P, stream);
    case 1: return launch_march_roles<Cfg<NSRC, false, false, true, NOSSIM>>(P, stream);
    case 2: return launch_march_roles<Cfg<NSRC, false, true, false, NOSSIM>>(P, stream);
    case 3: return launch_march_roles<Cfg<NSRC, false, true, true, NOSSIM>>(P, stream);
    case 4: return launch_march_roles<Cfg<NSRC, true, false, false, NOSSIM>>(P, stream);
    case 5: return launch_march_roles<Cfg<NSRC, true, false, true, NOSSIM>>(P, stream);
    case 6: return launch_march_roles<Cfg<NSRC, true, true, false, NOSSIM>>(P, stream);
    default: return launch_march_roles<Cfg<NSRC, true, true, true, NOSSIM>>(P, stream);
  }
}
template <int NSRC>
static cudaError_t launch_march_ns(const Params& P, cudaStream_t stream) {
  return P.no_ssim ? launch_march_n<NSRC, true>(P, stream) : launch_march_n<NSRC, false>(P, stream);
}
template <int NSRC>
static void launch_identity_ns(const Params& P, int grid, cudaStream_t stream) {
  {
    // TMA-staged form: production-sized images whose row pitch is a multiple of 16 bytes, base pointers 16-byte
    // aligned (cuTensorMapEncodeTiled's requirements).  MD2_IDENTITY_TMA=0 disables it.
    static const bool tma_on = !(getenv("MD2_IDENTITY_TMA") && atoi(getenv("MD2_IDENTITY_TMA")) == 0);
    uintptr_t bits = (uintptr_t)P.tgt;
    for (int f = 0; f < NSRC; ++f) bits |= (uintptr_t)P.src[f];
    if (tma_on && !P.tgt8 && pack2_on() && (bits & 15) == 0 && P.W % 4 == 0 && P.W >= kTmaBoxW && P.H >= kTmaBoxH) {
      IdTensorMaps maps;
      bool ok = make_image_map(&maps.img[0], P.tgt, P.B, P.H, P.W);
      for (int f = 0; f < NSRC && ok; ++f) ok = make_image_map(&maps.img[1 + f], P.src[f], P.B, P.H, P.W);
      for (int f = NSRC; f < kMaxSrc; ++f) maps.img[1 + f] = maps.img[0];
      // the dynamic shared-memory limit is set once per instantiation and its result kept: if the attribute (or a
      // tensor map) cannot be had, the register-marching form below runs instead - same results, ~10 % slower
      static const cudaError_t attr_ssim =
          cudaFuncSetAttribute(md2_identity_tma<NSRC, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tma_smem_bytes(NSRC));
      static const cudaError_t attr_l1 =
          cudaFuncSetAttribute(md2_identity_tma<NSRC, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tma_smem_bytes(NSRC));
      if (ok && (P.no_ssim ? attr_l1 : attr_ssim) == cudaSuccess) {
        const dim3 g((P.W + kTmaCols - 1) / kTmaCols, (P.H + kTmaRows - 1) / kTmaRows, P.B);
        const int smem = tma_smem_bytes(NSRC);
        if (P.no_ssim) md2_identity_tma<NSRC, true><<<g, kTmaCols, smem, stream>>>(P, maps);
        else md2_identity_tma<NSRC, false><<<g, kTmaCols, smem, stream>>>(P, maps);
        return;
      }
      static bool warned = false;
      if (!warned && getenv("MD2_VERBOSE")) {
        warned = true;
        fprintf(stderr, "md2: TMA-staged identity pass unavailable (tensor map %s, attribute %s): register-marching form\n",
                ok ? "ok" : "failed", cudaGetErrorString(P.no_ssim ? attr_l1 : attr_ssim));
      }
    }
  }
  if constexpr (NSRC == 2) {
    if (pack2_on()) {      // the identity pass is forward-only: packed form unless MD2_PACK2=off
      if (P.no_ssim) md2_identity2<true><<<grid, kThreads, 0, stream>>>(P);
      else md2_identity2<false><<<grid, kThreads, 0, stream>>>(P);
      return;
    }
  }
  if (P.no_ssim) md2_identity<NSRC, true><<<grid, kThreads, 0, stream>>>(P);
  else md2_identity<NSRC, false><<<grid, kThreads, 0, stream>>>(P);
}

// optional CUDA events recorded around the marching kernel (bench.py roofline leg)
static cudaEvent_t g_prof_ev[2] = {nullptr, nullptr};
static bool g_prof_on = false;

cudaError_t profile_enable(bool on) {
  if (on && !g_prof_ev[0]) {
    cudaError_t e = cudaEventCreate(&g_prof_ev[0]);
    if (e != cudaSuccess) return e;
    e = cudaEventCreate(&g_prof_ev[1]);
    if (e != cudaSuccess) return e;
  }
  g_prof_on = on;
  return cudaSuccess;
}
cudaError_t profile_march_ms(float* ms) {
  if (!g_prof_ev[0]) return cudaErrorNotReady;
  cudaError_t e = cudaEventSynchronize(g_prof_ev[1]);
  if (e != cudaSuccess) return e;
  return cudaEventElapsedTime(ms, g_prof_ev[0], g_prof_ev[1]);
}

// side stream + events (per device) used to overlap the small smoothness kernels with the
// identity / marching kernels; fork/join with events so that the caller's stream semantics
// (and CUDA-graph capture of the caller's stream) are preserved
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  cudaStream_t stream2 = nullptr;      // depth planes (md2_depth_up), beside the identity pass and the smoothness kernels
  cudaEvent_t join2 = nullptr;
};
static SideStream g_side[64];
static std::mutex g_side_mu;

// one side stream + event pair per device, created under a lock, all or nothing (a failed creation leaves the slot
// empty, so that the next call tries again instead of running with null events)
static cudaError_t get_side(SideStream** out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
  std::lock_guard<std::mutex> lock(g_side_mu);
  SideStream& s = g_side[dev];
  if (!s.stream) {
    SideStream n;
    if ((e = cudaStreamCreateWithFlags(&n.stream, cudaStreamNonBlocking)) == cudaSuccess &&
        (e = cudaStreamCreateWithFlags(&n.stream2, cudaStreamNonBlocking)) == cudaSuccess &&
        (e = cudaEventCreateWithFlags(&n.fork, cudaEventDisableTiming)) == cudaSuccess &&
        (e = cudaEventCreateWithFlags(&n.join2, cudaEventDisableTiming)) == cudaSuccess)
      e = cudaEventCreateWithFlags(&n.join, cudaEventDisableTiming);
    if (e != cudaSuccess) {
      if (n.join) cudaEventDestroy(n.join);
      if (n.join2) cudaEventDestroy(n.join2);
      if (n.stream2) cudaStreamDestroy(n.stream2);
      if (n.fork) cudaEventDestroy(n.fork);
      if (n.stream) cudaStreamDestroy(n.stream);
      return e;
    }
    s = n;
  }
  *out = &s;
  return cudaSuccess;
}

// uint8 entry (md2_tensors::target_u8 ...): every frame and pyramid level converted once to planar float (x / 255,
// bit-identical to torchvision's ToTensor) - one thread per pixel, three coalesced byte reads, three coalesced stores
__global__ void __launch_bounds__(256) md2_u8_to_f32(Params P) {
  const int img = blockIdx.z, b = blockIdx.y;
  const int nfull = 1 + P.nsrc;
  const int s = img < nfull ? 0 : img - nfull + P.up0;          // colour slots of level >= 1 (level 0 = the target)
  const int lv = img < nfull ? 0 : P.lvl[s];
  const int plane = (P.H >> lv) * (P.W >> lv);
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= plane) return;
  const unsigned char* in = img == 0 ? P.tgt8 : (img < nfull ? P.src8[img - 1] : P.color8[s]);
  float* out = img < nfull ? P.cvt_img[img] : P.cvt_col[s];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const size_t o = P.u8_hwc ? ((size_t)b * plane + p) * 3 + c : ((size_t)b * 3 + c) * plane + p;
    out[((size_t)b * 3 + c) * plane + p] = u8_unit(__ldg(in + o));
  }
}

// bf16 / fp16 leaves (md2_problem::*_dtype, planned by fill_widen): every reduced-precision disparity, mask and pose
// leaf widened exactly to fp32 in workspace, one launch for all of them (blockIdx.y = job).  It runs on the caller's
// stream before anything else, so the prologue, the side-stream kernels and the marching kernel all read fp32 copies.
__global__ void __launch_bounds__(256) md2_widen(Widen Wd) {
  const WidenJob& j = Wd.job[blockIdx.y];
  const long long step = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < j.n; i += step) {
    const long long si = j.row ? (i / j.row) * j.stride + i % j.row : i;
    j.dst[i] = j.dtype == MD2_DTYPE_BF16 ? __bfloat162float(((const __nv_bfloat16*)j.src)[si])
                                         : __half2float(((const __half*)j.src)[si]);
  }
}

static cudaError_t launch_float_entry(const Params& P, cudaStream_t stream);

// The fork / join events and the side streams are shared by every call on a device: the enqueue of one call (a few
// dozen microseconds of host time) runs under a lock, so that calls issued from several host threads - on the same or on
// different streams - cannot interleave their event records and waits.  The GPU work itself is not serialised by this.
static std::mutex g_enqueue_mu;

cudaError_t launch_view_synthesis_loss(const Params& P, const Widen& Wd, cudaStream_t stream) {
  std::lock_guard<std::mutex> enqueue_lock(g_enqueue_mu);
  if (Wd.n > 0) {
    long long bx = (Wd.max_n + 255) / 256;
    if (bx > 1184) bx = 1184;                     // 8 blocks per SM, grid-stride beyond
    md2_widen<<<dim3((unsigned)bx, Wd.n), 256, 0, stream>>>(Wd);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
#ifndef MD2_DBG_DEVICE
  static const bool cvt_on = !(getenv("MD2_U8_CONVERT") && atoi(getenv("MD2_U8_CONVERT")) == 0);
  if (P.tgt8 && cvt_on) {
    dim3 grid((P.H * P.W + 255) / 256, P.B, 1 + P.nsrc + (P.S - P.up0));
    md2_u8_to_f32<<<grid, 256, 0, stream>>>(P);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    Params Q = P;
    Q.tgt = P.cvt_img[0]; Q.tgt8 = nullptr;
    for (int f = 0; f < P.nsrc; ++f) { Q.src[f] = P.cvt_img[1 + f]; Q.src8[f] = nullptr; }
    for (int s2 = 0; s2 < P.S; ++s2) { Q.color[s2] = P.lvl[s2] == 0 ? P.cvt_img[0] : P.cvt_col[s2]; Q.color8[s2] = nullptr; }
    return launch_float_entry(Q, stream);
  }
#endif
  return launch_float_entry(P, stream);
}

static cudaError_t launch_float_entry(const Params& P, cudaStream_t stream) {
  cudaError_t e;
  SideStream* side = nullptr;
  if ((e = get_side(&side)) != cudaSuccess) return e;
  md2_prologue<<<4, 256, 0, stream>>>(P);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if (P.posecnn) {
    dim3 grid(16, P.B, P.S);
    md2_updisp_sum<<<grid, 256, 0, stream>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    md2_posecnn_setup<<<P.B, 32, 0, stream>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  if (P.pmask_on) {
    dim3 grid(16, P.B * P.nsrc, P.S);
    md2_pmask_up<<<grid, 256, 0, stream>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  // ---- fork: disparity means + smoothness on the side stream
  if ((e = cudaEventRecord(side->fork, stream)) != cudaSuccess) return e;
  if ((e = cudaStreamWaitEvent(side->stream, side->fork, 0)) != cudaSuccess) return e;
  {
    const int n0 = P.H * P.W;
    dim3 grid((n0 + 256 * 8 - 1) / (256 * 8), P.B, P.S);
    md2_disp_mean<<<grid, 256, 0, side->stream>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    int sjobs = 0;
    for (int s = 0; s < P.S; ++s) sjobs += smooth_bands(P.W >> P.lvl[s]) * smooth_segs(P.H >> P.lvl[s]) * P.B;
    md2_smooth<<<(sjobs + kSmoothWarps - 1) / kSmoothWarps, kSmoothWarps * 32, 0, side->stream>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    md2_smooth_scalars<<<(P.S * P.B + 63) / 64, 64, 0, side->stream>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  if ((e = cudaEventRecord(side->join, side->stream)) != cudaSuccess) return e;
  // ---- main stream: depth planes (role kernels), (identity + re-layout) or re-layout alone, then the marching kernel
  // (measured at 640x192 x 12: on the caller's stream in front of the identity pass the 12 us of md2_depth_up are
  // fully exposed; on the smoothness side stream they are too, that stream being as long as the identity pass)
  const bool zup = P.S > P.up0;
  if (zup) {
    if ((e = cudaStreamWaitEvent(side->stream2, side->fork, 0)) != cudaSuccess) return e;
    dim3 grid((P.W + kDupCols - 1) / kDupCols, (P.H + kDupRows - 1) / kDupRows, P.B * (P.S - P.up0));
    md2_depth_up<<<grid, 256, 0, side->stream2>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if ((e = cudaEventRecord(side->join2, side->stream2)) != cudaSuccess) return e;
  }
  if (P.automask) {
    const int jobs = P.B * P.nseg_id * P.nband_id;
    const int grid = (jobs + kWarpsPerCta - 1) / kWarpsPerCta;
    switch (P.nsrc) {
      case 1: launch_identity_ns<1>(P, grid, stream); break;
      case 2: launch_identity_ns<2>(P, grid, stream); break;
      case 3: launch_identity_ns<3>(P, grid, stream); break;
      case 4: launch_identity_ns<4>(P, grid, stream); break;
      default: return cudaErrorInvalidValue;
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  } else {
    dim3 grid((P.H * P.W + 255) / 256, P.B, 1 + P.nsrc);
    md2_pack<<<grid, 256, 0, stream>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  // ---- join: the marching kernel finishes grad_disp_0 and needs the smoothness sums
  if ((e = cudaStreamWaitEvent(stream, side->join, 0)) != cudaSuccess) return e;
  if (zup && (e = cudaStreamWaitEvent(stream, side->join2, 0)) != cudaSuccess) return e;
  // the tie-break noise may have been drawn on another stream (md2_tensors.noise_ready_event): first read is here
  if (P.noise_event && (e = cudaStreamWaitEvent(stream, (cudaEvent_t)P.noise_event, 0)) != cudaSuccess) return e;
  if (g_prof_on) cudaEventRecord(g_prof_ev[0], stream);
  switch (P.nsrc) {
    case 1: e = launch_march_ns<1>(P, stream); break;
    case 2: e = launch_march_ns<2>(P, stream); break;
    case 3: e = launch_march_ns<3>(P, stream); break;
    case 4: e = launch_march_ns<4>(P, stream); break;
    default: e = cudaErrorInvalidValue; break;
  }
  if (e != cudaSuccess) return e;
  if (g_prof_on) cudaEventRecord(g_prof_ev[1], stream);
  if (P.posecnn && P.want_grad) {
    md2_posecnn_final<<<P.B, 256, 0, stream>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  if (P.pmask_on && P.want_grad) {
    dim3 grid((P.H * P.W + 255) / 256, P.B * P.nsrc, P.S);
    md2_pmask_grad<<<grid, 256, 0, stream>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  // ---- scales >= 1: up-sampling adjoint + smoothness adjoint; losses; grad_T
  {
    int blocks = 0;
    if (P.want_grad)
      for (int s = P.up0; s < P.S; ++s)
        blocks += final_tiles_x(P.W >> P.lvl[s], 1 << P.lvl[s]) * final_tiles_y(P.H >> P.lvl[s], 1 << P.lvl[s]) * P.B;
    md2_final<<<blocks > 0 ? blocks : 1, kFinalThreads, 0, stream>>>(P);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  return cudaSuccess;
}

#if defined(MD2_DBG_DEVICE) || defined(MD2_BOUNDS_CHECK)
// debug build only (include/md2_debug.h)
cudaError_t debug_set_sink(const DebugSink* host_copy) {
#ifdef MD2_DBG_DEVICE
  DebugSink z;
  memset(&z, 0, sizeof(z));
  return cudaMemcpyToSymbol(g_dbg_sink, host_copy ? host_copy : &z, sizeof(DebugSink));
#else
  (void)host_copy;
  return cudaErrorNotSupported;
#endif
}
__global__ void md2_oob_rw(unsigned long long* out, int reset) {
#if defined(MD2_BOUNDS_CHECK)
  if (out) *out = g_oob_count;
  if (reset) g_oob_count = 0ULL;
#else
  if (out) *out = ~0ULL;
#endif
}
cudaError_t debug_oob_count(unsigned long long* count, int reset) {
  unsigned long long* d = nullptr;
  cudaError_t e = cudaMalloc((void**)&d, sizeof(*d));
  if (e != cudaSuccess) return e;
  md2_oob_rw<<<1, 1>>>(d, reset);
  e = cudaMemcpy(count, d, sizeof(*d), cudaMemcpyDeviceToHost);
  cudaFree(d);
  return e;
}
#endif

}  // namespace md2
