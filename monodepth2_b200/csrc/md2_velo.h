// md2_velo.h - the per-point and per-pixel arithmetic of md2_velo_depth, shared by the CUDA kernels and a g++ build
// (tests/test_velo_depth.py compiles it on the host and holds it to numpy and scipy.ndimage).
//
// Every double operation is spelled with an explicit rounding (no fused multiply-add on the device) so that both
// compilers evaluate the same sequence of IEEE operations.
#ifndef MD2_VELO_H_
#define MD2_VELO_H_

#include <math.h>

#ifdef __CUDACC__
#define MD2_HD __host__ __device__ __forceinline__
#else
#define MD2_HD inline
#endif

#ifdef __CUDA_ARCH__
#define MD2_DMUL(a, b) __dmul_rn((a), (b))
#define MD2_DADD(a, b) __dadd_rn((a), (b))
#else
#define MD2_DMUL(a, b) ((a) * (b))
#define MD2_DADD(a, b) ((a) + (b))
#endif

// Source index of output index `o` of skimage.transform.resize(order=0) along an axis of n_in -> n_out, i.e.
// scipy.ndimage.zoom(grid_mode=True, mode='grid-constant', order=0): the coordinate (o + 0.5) * (n_in / n_out) - 0.5,
// in float64 and in that order, rounded by floor(c + 0.5).  The exact .5 ties this meets (370 -> 375 rows 37, 112, ...)
// are decided by the float64 rounding of n_in / n_out, so no other expression form agrees.  -1: outside the input
// (cval 0).
// md2_velo_zoom is the factor, md2_velo_nearest_src_z the index from it (the kernel computes the factor once per job).
MD2_HD double md2_velo_zoom(int n_in, int n_out) { return (double)n_in / (double)n_out; }
MD2_HD int md2_velo_nearest_src_z(int o, int n_in, double zoom) {
  const double c = MD2_DADD(MD2_DADD(MD2_DMUL(MD2_DADD((double)o, 0.5), zoom), -0.5), 0.5);
  const double f = floor(c);
  return (f >= 0.0 && f < (double)n_in) ? (int)f : -1;
}
MD2_HD int md2_velo_nearest_src(int o, int n_in, int n_out) {
  return md2_velo_nearest_src_z(o, n_in, md2_velo_zoom(n_in, n_out));
}

// generate_depth_map for one point (x, y, z) of a scan (kitti_utils.py): (u', v', w) = P (x, y, z, 1) in float64,
// u = u' / w, v = v' / w, col = rint(u) - 1, row = rint(v) - 1 (np.round rounds half to even); the point lands when
// x >= 0 and (row, col) is inside height x width (a NaN or inf from w == 0 fails the tests).  Writes the pixel and the
// float64 value it stores (w, or x with vel_depth) and returns whether it lands.
MD2_HD bool md2_velo_project(const double* P, float x, float y, float z, int height, int width, int vel_depth,
                             int* row, int* col, double* value) {
  if (!(x >= 0.0f)) return false;
  const double X = x, Y = y, Z = z;
  const double up = MD2_DADD(MD2_DADD(MD2_DADD(MD2_DMUL(P[0], X), MD2_DMUL(P[1], Y)), MD2_DMUL(P[2], Z)), P[3]);
  const double vp = MD2_DADD(MD2_DADD(MD2_DADD(MD2_DMUL(P[4], X), MD2_DMUL(P[5], Y)), MD2_DMUL(P[6], Z)), P[7]);
  const double w = MD2_DADD(MD2_DADD(MD2_DADD(MD2_DMUL(P[8], X), MD2_DMUL(P[9], Y)), MD2_DMUL(P[10], Z)), P[11]);
  const double c = rint(up / w) - 1.0;
  const double r = rint(vp / w) - 1.0;
  if (!(c >= 0.0 && r >= 0.0 && c < (double)width && r < (double)height)) return false;
  *row = (int)r;
  *col = (int)c;
  *value = vel_depth ? X : w;
  return true;
}

// depth[depth < 0] = 0 on the float64 value, then the float32 rounding of MonoDataset.__getitem__.  Rounding is
// monotone, so a minimum over rounded values is the rounded minimum.  A zero is always +0.0: the reference keeps a
// -0.0 (a velodyne x of -0.0 under vel_depth) through some of numpy's reductions and clips and not others.
MD2_HD float md2_velo_store(double v) { return v > 0.0 ? (float)v : 0.0f; }

#endif  // MD2_VELO_H_
