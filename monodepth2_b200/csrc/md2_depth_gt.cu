// md2_depth_gt.cu - KITTI raw depth_gt on the GPU, from the velodyne scan.
//
// The reference builds depth_gt on the host for every sample (KITTIRAWDataset.get_depth, datasets/kitti_dataset.py;
// kitti_utils.py generate_depth_map): it projects the scan with P_velo2im in float64, writes each landing point's depth into the
// native map (the last point at a pixel wins), then, for every group of points sharing the reference's linear index
// sub2ind = row * (W - 1) + col - 1, writes the group's minimum at the pixel of its first point, clamps negatives to 0,
// resizes to full_res_shape with skimage's order-0 resize and flips.  sub2ind is off by one row stride, so besides equal
// pixels it also makes (r, W-1) and (r+1, 0) one group; those are its only extra collisions, so a group is one pixel
// plus at most that partner.
//
// Here that is three launches over every sample of a batch:
//   clear   - zero each sample's native cells (12 B per native pixel);
//   scatter - one thread per point: project and round (md2_velo.h), then per landing pixel atomicMax of the point index
//             (the last writer), atomicMin of the index (the first) and atomicMin of the float32 value as an
//             order-preserving uint - all three kept as maxima of encodings whose empty state is 0;
//   gather  - one thread per output pixel: flip, the nearest source pixel (md2_velo.h), and the rule above resolved from
//             that pixel's cell and its partner's; a last-writer value is recomputed from its point.
// The native map is never written.  Atomics of max/min are order-independent, so the result is bitwise reproducible.
// Grids depend only on the job count and the output size, so one CUDA graph serves batches of any scans.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/md2_loss.h"
#include "md2_velo.h"

namespace {

struct VeloCell {
  unsigned last;    // 1 + index of the last point, 0: empty
  unsigned first;   // ~index of the first point (atomicMax of ~i = atomicMin of i)
  unsigned vmin;    // ~order(value) of the smallest value
};
static_assert(sizeof(VeloCell) == 12, "12 bytes per native pixel");

constexpr int kThreads = 256;
constexpr int kBlocksTotal = 148 * 8;   // per launch of the clear and scatter passes, shared out among the jobs

// the largest native extent of an axis of n_out output pixels the ABI accepts (native / out < 1.25)
inline long long max_native(int n_out) { return (5LL * n_out - 1) / 4; }
inline size_t cells_per_job(int out_h, int out_w) { return (size_t)max_native(out_h) * (size_t)max_native(out_w); }

__device__ __forceinline__ unsigned order_f32(float f) {
  const unsigned b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float unorder_f32(unsigned o) {
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

__global__ void __launch_bounds__(kThreads) md2_velo_clear(const md2_velo_job* __restrict__ jobs, VeloCell* cells,
                                                           size_t slot) {
  const md2_velo_job& j = jobs[blockIdx.y];
  unsigned* c = reinterpret_cast<unsigned*>(cells + slot * blockIdx.y);
  const long long n = 3LL * j.height * j.width;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kThreads) c[i] = 0u;
}

__global__ void __launch_bounds__(kThreads) md2_velo_scatter(const unsigned char* __restrict__ scans,
                                                             const md2_velo_job* __restrict__ jobs, VeloCell* cells,
                                                             size_t slot) {
  const md2_velo_job& j = jobs[blockIdx.y];
  const float4* pts = reinterpret_cast<const float4*>(scans + j.offset);
  VeloCell* c = cells + slot * blockIdx.y;
  const int n = j.n_points, H = j.height, W = j.width, vel = j.vel_depth;
  double P[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) P[k] = j.P[k];
  for (int i = blockIdx.x * kThreads + threadIdx.x; i < n; i += gridDim.x * kThreads) {
    const float4 p = __ldg(pts + i);
    int row, col;
    double v;
    if (!md2_velo_project(P, p.x, p.y, p.z, H, W, vel, &row, &col, &v)) continue;
    VeloCell* cell = c + (size_t)row * W + col;
    atomicMax(&cell->last, (unsigned)i + 1u);
    atomicMax(&cell->first, ~(unsigned)i);
    atomicMax(&cell->vmin, ~order_f32(md2_velo_store(v)));
  }
}

__global__ void __launch_bounds__(kThreads) md2_velo_gather(const unsigned char* __restrict__ scans,
                                                            const md2_velo_job* __restrict__ jobs,
                                                            const VeloCell* __restrict__ cells, size_t slot,
                                                            float* __restrict__ out, int out_h, int out_w) {
  // a block is part of one output row of one job: its source row and the column factor are computed once
  __shared__ int s_sr;
  __shared__ double s_zoom_w;
  const int y = blockIdx.y;
  const md2_velo_job& j = jobs[blockIdx.z];
  const int H = j.height, W = j.width;
  if (threadIdx.x == 0) {
    s_sr = md2_velo_nearest_src(y, H, out_h);
    s_zoom_w = md2_velo_zoom(W, out_w);
  }
  __syncthreads();
  const int x = blockIdx.x * kThreads + threadIdx.x;
  if (x >= out_w) return;
  float d = 0.0f;
  const int sr = s_sr;                                                       // resize first, then np.fliplr
  const int sc = md2_velo_nearest_src_z(j.flip ? out_w - 1 - x : x, W, s_zoom_w);
  if (sr >= 0 && sc >= 0) {
    const VeloCell* c = cells + slot * blockIdx.z;
    const long long p = (long long)sr * W + sc;
    const VeloCell a = c[p];
    if (a.last != 0u) {
      VeloCell b = {0u, 0u, 0u};                                             // the sub2ind partner, if any
      if (sc == W - 1 && sr + 1 < H) b = c[p + 1];                           // (sr, W-1) ~ (sr+1, 0)
      else if (sc == 0 && sr > 0) b = c[p - 1];                              // (sr, 0) ~ (sr-1, W-1)
      const unsigned fa = ~a.first, la = a.last - 1u;
      const bool dup = fa != la || b.last != 0u;                             // the group holds more than one point
      if (dup && (b.last == 0u || fa < ~b.first)) {
        d = unorder_f32(min(~a.vmin, ~b.vmin));                              // min over the group, at its first point
      } else {
        const float4 q = __ldg(reinterpret_cast<const float4*>(scans + j.offset) + la);
        double P[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) P[k] = j.P[k];
        int row, col;
        double v = 0.0;
        md2_velo_project(P, q.x, q.y, q.z, H, W, j.vel_depth, &row, &col, &v);   // the last writer's value
        d = md2_velo_store(v);
      }
    }
  }
  out[((size_t)blockIdx.z * out_h + y) * out_w + x] = d;
}

}  // namespace

extern "C" {

int md2_velo_depth_scratch_bytes(int n_jobs, int out_h, int out_w, size_t* bytes) {
  if (!bytes || n_jobs < 1 || out_h < 1 || out_w < 1) return MD2_ERR_INVALID_ARGUMENT;
  *bytes = (size_t)n_jobs * cells_per_job(out_h, out_w) * sizeof(VeloCell);
  return MD2_OK;
}

int md2_velo_depth(const unsigned char* scans, size_t scans_bytes, const md2_velo_job* jobs, const md2_velo_job* jobs_dev,
                   int n_jobs, float* out, int out_h, int out_w, void* scratch, size_t scratch_bytes, void* stream) {
  if (!scans || !jobs || !jobs_dev || !out || n_jobs < 1 || out_h < 1 || out_w < 1) return MD2_ERR_INVALID_ARGUMENT;
  if (n_jobs > 65535 || out_h > 65535) return MD2_ERR_UNSUPPORTED;
  for (int i = 0; i < n_jobs; ++i) {
    const md2_velo_job& j = jobs[i];
    if (j.n_points < 0 || j.height < 1 || j.width < 1) return MD2_ERR_INVALID_ARGUMENT;
    if (j.offset < 0 || (size_t)j.offset > scans_bytes || (scans_bytes - (size_t)j.offset) / 16 < (size_t)j.n_points)
      return MD2_ERR_INVALID_ARGUMENT;                 // would read outside `scans`
    if (((uintptr_t)scans + (uintptr_t)j.offset) % 16 != 0) return MD2_ERR_INVALID_ARGUMENT;
    // skimage's anti-aliasing filter is the identity only below a factor of 1.25; with a width of 1 sub2ind makes
    // every pixel one group
    if (j.height > max_native(out_h) || j.width > max_native(out_w) || j.width < 2) return MD2_ERR_UNSUPPORTED;
  }
  const size_t slot = cells_per_job(out_h, out_w);
  if (!scratch || scratch_bytes < (size_t)n_jobs * slot * sizeof(VeloCell)) return MD2_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t s = (cudaStream_t)stream;
  VeloCell* cells = (VeloCell*)scratch;
  const dim3 spread((kBlocksTotal + n_jobs - 1) / n_jobs, n_jobs);
  md2_velo_clear<<<spread, kThreads, 0, s>>>(jobs_dev, cells, slot);
  md2_velo_scatter<<<spread, kThreads, 0, s>>>(scans, jobs_dev, cells, slot);
  md2_velo_gather<<<dim3((out_w + kThreads - 1) / kThreads, out_h, n_jobs), kThreads, 0, s>>>(scans, jobs_dev, cells,
                                                                                             slot, out, out_h, out_w);
  return cudaGetLastError() == cudaSuccess ? MD2_OK : MD2_ERR_CUDA;
}

}  // extern "C"
