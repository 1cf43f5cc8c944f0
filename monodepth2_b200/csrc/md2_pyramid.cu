// md2_pyramid.cu - colour pyramid on the GPU: Pillow's uint8 LANCZOS resize, byte for byte.
//
// The reference builds ("color", f, s) on the host, per frame and per sample, with torchvision
// transforms.Resize(..., interpolation=Image.ANTIALIAS) on PIL images: scale 0 from the native frame,
// scale i from scale i-1 (/root/reference/datasets/mono_dataset.py:57,82-86,98-103), i.e.
// PIL.Image.resize(size, LANCZOS).  Pillow (src/libImaging/Resample.c) does a separable two-pass resample in
// 8-bit fixed point: precompute_coeffs (double), normalize_coeffs_8bpc (22-bit integers), horizontal pass
// into a uint8 temporary, then the vertical pass; each output = clip8((2^21 + sum k_i * in_i) >> 22).
// The coefficient tables are built on the HOST with the same double arithmetic (libm sin) when the plan is
// created and uploaded once; the two passes are integer kernels, so the result is bit-identical to Pillow's
// (tests/test_pyramid.py: against oracle/pillow_resize.py and against the installed Pillow).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include <vector>

#include "../../include/md2_loss.h"

namespace {

constexpr int kPrecisionBits = 32 - 8 - 2;

double sinc_filter(double x) {
  if (x == 0.0) return 1.0;
  x = x * M_PI;
  return sin(x) / x;
}
double lanczos_filter(double x) {
  /* truncated sinc */
  if (-3.0 <= x && x < 3.0) return sinc_filter(x) * sinc_filter(x / 3);
  return 0.0;
}

// Resample.c precompute_coeffs + normalize_coeffs_8bpc for the whole-image box
struct Coeffs {
  int ksize = 0;
  std::vector<int> bounds;   // out_size x (xmin, count)
  std::vector<int> kk;       // out_size x ksize
};
Coeffs precompute(int in_size, int out_size) {
  Coeffs c;
  double scale, filterscale;
  filterscale = scale = (double)in_size / out_size;
  if (filterscale < 1.0) filterscale = 1.0;
  const double support = 3.0 * filterscale;
  c.ksize = (int)ceil(support) * 2 + 1;
  c.bounds.assign((size_t)out_size * 2, 0);
  c.kk.assign((size_t)out_size * c.ksize, 0);
  std::vector<double> w(c.ksize);
  const double ss = 1.0 / filterscale;
  for (int xx = 0; xx < out_size; ++xx) {
    const double center = (xx + 0.5) * scale;
    double ww = 0.0;
    int xmin = (int)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(center + support + 0.5);
    if (xmax > in_size) xmax = in_size;
    xmax -= xmin;
    for (int x = 0; x < xmax; ++x) {
      w[x] = lanczos_filter((x + xmin - center + 0.5) * ss);
      ww += w[x];
    }
    for (int x = 0; x < xmax; ++x) {
      const double k = (ww != 0.0) ? w[x] / ww : w[x];
      c.kk[(size_t)xx * c.ksize + x] = (k < 0) ? (int)(-0.5 + k * (1 << kPrecisionBits)) : (int)(0.5 + k * (1 << kPrecisionBits));
    }
    c.bounds[2 * xx] = xmin;
    c.bounds[2 * xx + 1] = xmax;
  }
  return c;
}

__device__ __forceinline__ unsigned char clip8(int v) {
  v >>= kPrecisionBits;
  return (unsigned char)(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// Coefficient table of one resampled axis (device arrays from precompute).
struct Table {
  const int* bounds;
  const int* kk;
  int ksize;
};

// One separable pass.  AXIS 0: resample x (rows unchanged); AXIS 1: resample y.  Element (c, y, x) of an image at
// c*cs + y*ys + x*xs, HWC or CHW independently for input and output; output image b at b * 3 * out_h * out_w.
// Uniform batch (jobs == nullptr): input image b at b * in_img, of size (in_h, in_w), resampled with tables[0].
// Job list: the native size and the table come from jobs[b] (tables[jobs[b].size]); the horizontal pass reads the native
// frame at jobs[b].offset, mirrored when jobs[b].flip (column w-1-x, i.e. transpose(FLIP_LEFT_RIGHT) then resize), and
// writes rows [0, height) of an out_h-row temporary; the vertical pass reads that temporary at b * in_img.
template <int AXIS>
__global__ void md2_resample_u8(const unsigned char* __restrict__ in, unsigned char* __restrict__ out,
                                const md2_batch_job* __restrict__ jobs, const Table* __restrict__ tables, int batch,
                                int in_h, int in_w, int out_h, int out_w, long long in_img, int in_hwc, int out_hwc) {
  const long long n = (long long)batch * out_h * out_w;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int x = (int)(i % out_w);
  const int y = (int)((i / out_w) % out_h);
  const int b = (int)(i / ((long long)out_w * out_h));
  const unsigned char* src = in + (long long)b * in_img;
  int ih = in_h, iw = in_w, flip = 0, t = 0;
  if (jobs) {
    ih = __ldg(&jobs[b].height);
    t = __ldg(&jobs[b].size);
    if (AXIS == 0) {
      if (y >= ih) return;
      iw = __ldg(&jobs[b].width);
      flip = __ldg(&jobs[b].flip);
      src = in + __ldg(&jobs[b].offset);
    }
  }
  const long long ics = in_hwc ? 1 : (long long)ih * iw, ixs = in_hwc ? 3 : 1, iys = (long long)iw * ixs;
  const long long ocs = out_hwc ? 1 : (long long)out_h * out_w, oxs = out_hwc ? 3 : 1, oys = (long long)out_w * oxs;
  unsigned char* dst = out + (long long)b * 3 * out_h * out_w + y * oys + x * oxs;
  const int o = AXIS == 0 ? x : y;
  const int* bounds = tables[t].bounds;
  const int lo = __ldg(bounds + 2 * o), cnt = __ldg(bounds + 2 * o + 1);
  const int* k = tables[t].kk + (size_t)o * tables[t].ksize;
  int s0 = 1 << (kPrecisionBits - 1), s1 = s0, s2 = s0;
  const unsigned char* p = AXIS == 0 ? src + y * iys + (flip ? iw - 1 - lo : lo) * ixs : src + lo * iys + x * ixs;
  const long long step = AXIS == 0 ? (flip ? -ixs : ixs) : iys;
  for (int j = 0; j < cnt; ++j) {
    const int w = __ldg(k + j);
    s0 += (int)__ldg(p) * w;
    s1 += (int)__ldg(p + ics) * w;
    s2 += (int)__ldg(p + 2 * ics) * w;
    p += step;
  }
  dst[0] = clip8(s0);
  dst[ocs] = clip8(s1);
  dst[2 * ocs] = clip8(s2);
}

// ------------------------------------------------------------------ colour augmentation (SURVEY.md 8f-3)
// torchvision ColorJitter on PIL images as MonoDataset applies it (/root/reference/datasets/mono_dataset.py:60-70,
// 136,169-176): adjust_brightness / contrast / saturation = Pillow's Image.blend(degenerate, image, factor)
// (libImaging/Blend.c: in1 + alpha * (in2 - in1) in C float, truncated), the "L" conversion of Convert.c, and
// adjust_hue = RGB -> HSV -> h += shift (mod 256) -> RGB with Convert.c's float / double mix.  Every operation is
// written with explicit _rn intrinsics (no contraction) so that the bytes equal Pillow's; oracle/color_jitter.py is the
// restatement the tests hold this to (itself pinned against the installed Pillow, the HSV pair on all 2^24 colours).
struct Rgb8 { int r, g, b; };

__device__ __forceinline__ int cj_to_l(const Rgb8& c) { return (c.r * 19595 + c.g * 38470 + c.b * 7471 + 0x8000) >> 16; }

__device__ __forceinline__ int cj_blend1(int in1, int in2, float a, bool interp) {
  const float t = __fadd_rn((float)in1, __fmul_rn(a, (float)(in2 - in1)));
  if (interp) return (int)t;
  return t <= 0.0f ? 0 : (t >= 255.0f ? 255 : (int)t);
}
__device__ __forceinline__ Rgb8 cj_blend(const Rgb8& d, const Rgb8& c, float a) {
  const bool interp = a >= 0.0f && a <= 1.0f;
  Rgb8 o;
  o.r = cj_blend1(d.r, c.r, a, interp); o.g = cj_blend1(d.g, c.g, a, interp); o.b = cj_blend1(d.b, c.b, a, interp);
  return o;
}

__device__ __forceinline__ Rgb8 cj_hue(const Rgb8& c, int shift) {
  // rgb2hsv_row
  const int maxc = max(c.r, max(c.g, c.b)), minc = min(c.r, min(c.g, c.b));
  int uh = 0, us = 0;
  const int uv = maxc;
  if (minc != maxc) {
    const float cr = (float)(maxc - minc);
    const float sf = __fdiv_rn(cr, (float)maxc);
    const float rc = __fdiv_rn((float)(maxc - c.r), cr), gc = __fdiv_rn((float)(maxc - c.g), cr), bc = __fdiv_rn((float)(maxc - c.b), cr);
    float h;
    if (c.r == maxc) h = __fsub_rn(bc, gc);
    else if (c.g == maxc) h = __double2float_rn(__dsub_rn(__dadd_rn(2.0, (double)rc), (double)bc));
    else h = __double2float_rn(__dsub_rn(__dadd_rn(4.0, (double)gc), (double)rc));
    h = __double2float_rn(fmod(__dadd_rn(__ddiv_rn((double)h, 6.0), 1.0), 1.0));
    uh = min(max((int)__dmul_rn((double)h, 255.0), 0), 255);
    us = min(max((int)__dmul_rn((double)sf, 255.0), 0), 255);
  }
  uh = (uh + shift) & 255;
  // hsv2rgb
  Rgb8 o;
  if (us == 0) { o.r = o.g = o.b = uv; return o; }
  const double hf = __ddiv_rn(__dmul_rn((double)(float)uh, 6.0), 255.0);
  const int i = (int)floor(hf);
  const double f = (double)__double2float_rn(__dsub_rn(hf, (double)(float)i));
  const double fs = (double)__double2float_rn(__ddiv_rn((double)(float)us, 255.0));
  const double vf = (double)(float)uv;
  const int p = min(max((int)round(__dmul_rn(vf, __dsub_rn(1.0, fs))), 0), 255);
  const int q = min(max((int)round(__dmul_rn(vf, __dsub_rn(1.0, __dmul_rn(fs, f)))), 0), 255);
  const int t = min(max((int)round(__dmul_rn(vf, __dsub_rn(1.0, __dmul_rn(fs, __dsub_rn(1.0, f))))), 0), 255);
  switch (i % 6) {
    case 0: o.r = uv; o.g = t; o.b = p; break;
    case 1: o.r = q; o.g = uv; o.b = p; break;
    case 2: o.r = p; o.g = uv; o.b = t; break;
    case 3: o.r = p; o.g = q; o.b = uv; break;
    case 4: o.r = t; o.g = p; o.b = uv; break;
    default: o.r = uv; o.g = p; o.b = q; break;
  }
  return o;
}

// applies operations [from, to) of the image's order; `mean` is the contrast gray level (used when op 1 is in range)
__device__ __forceinline__ Rgb8 cj_apply(Rgb8 c, const md2_color_jitter& J, int from, int to, int mean) {
  for (int k = from; k < to; ++k) {
    const int op = J.order[k];
    if (op == 0) { const Rgb8 z = {0, 0, 0}; c = cj_blend(z, c, J.brightness); }
    else if (op == 1) { const Rgb8 m = {mean, mean, mean}; c = cj_blend(m, c, J.contrast); }
    else if (op == 2) { const int l = cj_to_l(c); const Rgb8 g = {l, l, l}; c = cj_blend(g, c, J.saturation); }
    else if (op == 3) c = cj_hue(c, J.hue_shift);
  }
  return c;
}
__device__ __forceinline__ int cj_contrast_pos(const md2_color_jitter& J) {
  for (int k = 0; k < 4; ++k) if (J.order[k] == 1) return k;
  return -1;
}
__device__ __forceinline__ Rgb8 cj_load(const unsigned char* in, long long n, int p, int plane, int hwc) {
  Rgb8 c;
  if (hwc) { const unsigned char* q = in + (n * plane + p) * 3; c.r = __ldg(q); c.g = __ldg(q + 1); c.b = __ldg(q + 2); }
  else { const unsigned char* q = in + n * 3 * plane + p; c.r = __ldg(q); c.g = __ldg(q + plane); c.b = __ldg(q + 2 * (long long)plane); }
  return c;
}

// The images of one jitter call: level s (s < n_levels) holds n_img images of plane[s] pixels starting at element off[s]
// of the input and of each output; image y of the grid is image y % n_img of level y / n_img.  The one-size entry is the
// case n_levels == 1.  Image i's parameter row is jobs[i].sample (job list) or i.
struct CjImages {
  int n_img, n_levels;
  int plane[MD2_MAX_SCALES];
  long long off[MD2_MAX_SCALES];
};
struct CjImage {
  int level, i, plane;
  long long off;
};
__device__ __forceinline__ CjImage cj_image(const CjImages& im) {
  CjImage r;
  r.level = blockIdx.y / im.n_img;
  r.i = blockIdx.y - r.level * im.n_img;
#pragma unroll
  for (int l = 0; l < MD2_MAX_SCALES; ++l)          // a select, not a dynamic index (that would copy `im` to the stack)
    if (l == r.level) { r.plane = im.plane[l]; r.off = im.off[l]; }
  return r;
}

// pass 1 (only for images whose order contains contrast): sum of the "L" image after the operations in front of it
__global__ void __launch_bounds__(256) md2_cj_lsum(const unsigned char* in, const md2_color_jitter* params,
                                                    const md2_batch_job* jobs, unsigned long long* sums, CjImages im,
                                                    int hwc) {
  const CjImage g = cj_image(im);
  const md2_color_jitter J = params[jobs ? jobs[g.i].sample : g.i];
  const int cp = cj_contrast_pos(J);
  if (cp < 0) return;
  unsigned int acc = 0;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < g.plane; p += gridDim.x * blockDim.x)
    acc += (unsigned)cj_to_l(cj_apply(cj_load(in + g.off, g.i, p, g.plane, hwc), J, 0, cp, 0));
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(sums + blockIdx.y, (unsigned long long)acc);
}

// pass 2: the whole chain; mean = int(sum / count + 0.5) in double, as ImageStat.Stat(...).mean does in Python.
// Writes the jittered bytes to out_u8 (one-size entry) or their ToTensor value x / 255 to out_aug (job list), and with
// out_color the unjittered ToTensor value.
__global__ void __launch_bounds__(256) md2_cj_apply(const unsigned char* in, unsigned char* out_u8, float* out_aug,
                                                     float* out_color, const md2_color_jitter* params,
                                                     const md2_batch_job* jobs, const unsigned long long* sums,
                                                     CjImages im, int hwc) {
  const CjImage g = cj_image(im);
  const md2_color_jitter J = params[jobs ? jobs[g.i].sample : g.i];
  const int mean = (int)(__dadd_rn(__ddiv_rn((double)sums[blockIdx.y], (double)g.plane), 0.5));
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < g.plane; p += gridDim.x * blockDim.x) {
    const Rgb8 x = cj_load(in + g.off, g.i, p, g.plane, hwc);
    const Rgb8 c = cj_apply(x, J, 0, 4, mean);
    if (out_u8) {
      unsigned char* q = out_u8 + g.off;
      if (hwc) { q += ((long long)g.i * g.plane + p) * 3; q[0] = (unsigned char)c.r; q[1] = (unsigned char)c.g; q[2] = (unsigned char)c.b; }
      else { q += (long long)g.i * 3 * g.plane + p; q[0] = (unsigned char)c.r; q[g.plane] = (unsigned char)c.g; q[2 * (long long)g.plane] = (unsigned char)c.b; }
    }
    const long long e = g.off + (long long)g.i * 3 * g.plane + p;    // CHW (the job list is NCHW)
    if (out_aug) {
      out_aug[e] = __fdiv_rn((float)c.r, 255.0f);
      out_aug[e + g.plane] = __fdiv_rn((float)c.g, 255.0f);
      out_aug[e + 2 * (long long)g.plane] = __fdiv_rn((float)c.b, 255.0f);
    }
    if (out_color) {
      out_color[e] = __fdiv_rn((float)x.r, 255.0f);
      out_color[e + g.plane] = __fdiv_rn((float)x.g, 255.0f);
      out_color[e + 2 * (long long)g.plane] = __fdiv_rn((float)x.b, 255.0f);
    }
  }
}

// grid of one jitter call: enough blocks for the largest plane (capped; both passes stride over the rest)
void cj_launch(const unsigned char* in, unsigned char* out_u8, float* out_aug, float* out_color, const md2_color_jitter* params,
               const md2_batch_job* jobs, unsigned long long* sums, const CjImages& im, int hwc, cudaStream_t s) {
  const int n = im.n_img * im.n_levels;
  const int bx = (im.plane[0] + 255) / 256;
  md2_cj_lsum<<<dim3(bx < 64 ? bx : 64, n), 256, 0, s>>>(in, params, jobs, sums, im, hwc);
  md2_cj_apply<<<dim3(bx < 128 ? bx : 128, n), 256, 0, s>>>(in, out_u8, out_aug, out_color, params, jobs, sums, im, hwc);
}

}  // namespace

namespace {

// the two device arrays of one axis's table (owned by the plan that made it)
struct AxisTable {
  int* bounds = nullptr;
  int* kk = nullptr;
  int ksize = 0;
};
bool upload(const std::vector<int>& v, int** d) {
  if (cudaMalloc((void**)d, v.size() * sizeof(int)) != cudaSuccess) { *d = nullptr; return false; }
  return cudaMemcpy(*d, v.data(), v.size() * sizeof(int), cudaMemcpyHostToDevice) == cudaSuccess;
}
bool make_axis(int in_size, int out_size, AxisTable* a) {
  const Coeffs c = precompute(in_size, out_size);
  a->ksize = c.ksize;
  return upload(c.bounds, &a->bounds) && upload(c.kk, &a->kk);
}
void free_axis(AxisTable* a) {
  cudaFree(a->bounds); cudaFree(a->kk);
  *a = AxisTable();
}
Table as_table(const AxisTable& a) { return Table{a.bounds, a.kk, a.ksize}; }

}  // namespace

struct md2_resize_plan {
  int in_h, in_w, out_h, out_w;
  AxisTable x, y;
  Table* tables;   // device: {x, y}
};

struct md2_batch_plan {
  int height, width, num_scales;
  int n_sizes, max_h;
  int size_h[MD2_BATCH_MAX_SIZES], size_w[MD2_BATCH_MAX_SIZES];
  AxisTable ax[MD2_BATCH_MAX_SIZES], ay[MD2_BATCH_MAX_SIZES];
  Table *tx, *ty;                              // device, MD2_BATCH_MAX_SIZES entries each: native w -> width, h -> height
  md2_resize_plan* level[MD2_MAX_SCALES];      // level s-1 -> level s, s >= 1
};

namespace {

// scratch of md2_batch_build_u8: contrast sums | resample temporary | uint8 levels (float colour only)
struct BatchScratch {
  size_t sums, tmp, levels, total;
};
BatchScratch batch_scratch(const md2_batch_plan* p, int n, int color_f32) {
  BatchScratch b;
  const size_t nn = (size_t)n;
  b.sums = (nn * p->num_scales * sizeof(unsigned long long) + 255) / 256 * 256;
  b.tmp = nn * 3 * p->max_h * p->width;                   // level 0's horizontal pass, native rows
  size_t planes = (size_t)p->height * p->width;
  for (int s = 1; s < p->num_scales; ++s) {
    const size_t lt = nn * 3 * (p->height >> (s - 1)) * (p->width >> s);   // md2_resize_scratch_bytes of level s
    if (lt > b.tmp) b.tmp = lt;
    planes += (size_t)(p->height >> s) * (p->width >> s);
  }
  b.tmp = (b.tmp + 255) / 256 * 256;
  b.levels = color_f32 ? nn * 3 * planes : 0;
  b.total = b.sums + b.tmp + b.levels;
  return b;
}

}  // namespace

extern "C" {

int md2_resize_plan_create(int in_h, int in_w, int out_h, int out_w, md2_resize_plan** plan) {
  if (!plan || in_h < 1 || in_w < 1 || out_h < 1 || out_w < 1) return MD2_ERR_INVALID_ARGUMENT;
  md2_resize_plan* p = (md2_resize_plan*)calloc(1, sizeof(md2_resize_plan));
  if (!p) return MD2_ERR_INVALID_ARGUMENT;
  p->in_h = in_h; p->in_w = in_w; p->out_h = out_h; p->out_w = out_w;
  const Table t[2] = {Table{}, Table{}};
  bool ok = make_axis(in_w, out_w, &p->x) && make_axis(in_h, out_h, &p->y) &&
            cudaMalloc((void**)&p->tables, sizeof(t)) == cudaSuccess;
  if (ok) {
    const Table h[2] = {as_table(p->x), as_table(p->y)};
    ok = cudaMemcpy(p->tables, h, sizeof(h), cudaMemcpyHostToDevice) == cudaSuccess;
  }
  if (!ok) {
    md2_resize_plan_destroy(p);
    return MD2_ERR_CUDA;
  }
  *plan = p;
  return MD2_OK;
}

void md2_resize_plan_destroy(md2_resize_plan* p) {
  if (!p) return;
  free_axis(&p->x); free_axis(&p->y); cudaFree(p->tables);
  free(p);
}

int md2_resize_scratch_bytes(const md2_resize_plan* p, int batch, size_t* bytes) {
  if (!p || !bytes || batch < 1) return MD2_ERR_INVALID_ARGUMENT;
  *bytes = (size_t)batch * 3 * p->in_h * p->out_w;     // the horizontal pass's uint8 temporary
  return MD2_OK;
}

int md2_resize_lanczos_u8(const md2_resize_plan* p, const unsigned char* in, unsigned char* out, void* scratch,
                          size_t scratch_bytes, int batch, int hwc, void* stream) {
  if (!p || !in || !out || batch < 1) return MD2_ERR_INVALID_ARGUMENT;
  cudaStream_t s = (cudaStream_t)stream;
  const bool need_x = p->in_w != p->out_w, need_y = p->in_h != p->out_h;
  if (need_x && need_y) {
    size_t need = 0;
    md2_resize_scratch_bytes(p, batch, &need);
    if (!scratch || scratch_bytes < need) return MD2_ERR_WORKSPACE_TOO_SMALL;
  }
  const unsigned char* cur = in;
  int cur_w = p->in_w;
  if (need_x) {
    unsigned char* dst = need_y ? (unsigned char*)scratch : out;
    const long long n = (long long)batch * p->in_h * p->out_w;
    md2_resample_u8<0><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(cur, dst, nullptr, p->tables, batch, p->in_h, p->in_w,
                                                                    p->in_h, p->out_w, 3LL * p->in_h * p->in_w, hwc, hwc);
    cur = dst;
    cur_w = p->out_w;
  }
  if (need_y) {
    const long long n = (long long)batch * p->out_h * p->out_w;
    md2_resample_u8<1><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(cur, out, nullptr, p->tables + 1, batch, p->in_h, cur_w,
                                                                    p->out_h, p->out_w, 3LL * p->in_h * cur_w, hwc, hwc);
  }
  if (!need_x && !need_y) {
    if (cudaMemcpyAsync(out, in, (size_t)batch * 3 * p->in_h * p->in_w, cudaMemcpyDeviceToDevice, s) != cudaSuccess)
      return MD2_ERR_CUDA;
  }
  return cudaGetLastError() == cudaSuccess ? MD2_OK : MD2_ERR_CUDA;
}

int md2_color_jitter_u8(const unsigned char* in, unsigned char* out, const md2_color_jitter* params, void* scratch,
                        size_t scratch_bytes, int n_images, int height, int width, int hwc, void* stream) {
  if (!in || !out || !params || n_images < 1 || height < 1 || width < 1) return MD2_ERR_INVALID_ARGUMENT;
  if (n_images > 65535) return MD2_ERR_UNSUPPORTED;
  if (!scratch || scratch_bytes < (size_t)n_images * sizeof(unsigned long long)) return MD2_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t s = (cudaStream_t)stream;
  unsigned long long* sums = (unsigned long long*)scratch;
  if (cudaMemsetAsync(sums, 0, (size_t)n_images * sizeof(unsigned long long), s) != cudaSuccess) return MD2_ERR_CUDA;
  CjImages im = {};
  im.n_img = n_images; im.n_levels = 1; im.plane[0] = height * width;
  cj_launch(in, out, nullptr, nullptr, params, nullptr, sums, im, hwc, s);
  return cudaGetLastError() == cudaSuccess ? MD2_OK : MD2_ERR_CUDA;
}

int md2_batch_plan_create(int height, int width, int num_scales, md2_batch_plan** plan) {
  if (!plan || num_scales < 1 || num_scales > MD2_MAX_SCALES || height < 1 || width < 1 ||
      (height >> (num_scales - 1)) < 1 || (width >> (num_scales - 1)) < 1)
    return MD2_ERR_INVALID_ARGUMENT;
  md2_batch_plan* p = (md2_batch_plan*)calloc(1, sizeof(md2_batch_plan));
  if (!p) return MD2_ERR_INVALID_ARGUMENT;
  p->height = height; p->width = width; p->num_scales = num_scales;
  *plan = p;                  // device tables are made when the first native size is added
  return MD2_OK;
}

void md2_batch_plan_destroy(md2_batch_plan* p) {
  if (!p) return;
  for (int i = 0; i < p->n_sizes; ++i) { free_axis(&p->ax[i]); free_axis(&p->ay[i]); }
  for (int s = 1; s < MD2_MAX_SCALES; ++s) md2_resize_plan_destroy(p->level[s]);
  cudaFree(p->tx); cudaFree(p->ty);
  free(p);
}

int md2_batch_plan_add_native_size(md2_batch_plan* p, int h, int w, int* index) {
  if (!p || !index || h < 1 || w < 1) return MD2_ERR_INVALID_ARGUMENT;
  for (int i = 0; i < p->n_sizes; ++i)
    if (p->size_h[i] == h && p->size_w[i] == w) { *index = i; return MD2_OK; }
  if (p->n_sizes == MD2_BATCH_MAX_SIZES) return MD2_ERR_UNSUPPORTED;
  if (!p->tx && cudaMalloc((void**)&p->tx, MD2_BATCH_MAX_SIZES * sizeof(Table)) != cudaSuccess) { p->tx = nullptr; return MD2_ERR_CUDA; }
  if (!p->ty && cudaMalloc((void**)&p->ty, MD2_BATCH_MAX_SIZES * sizeof(Table)) != cudaSuccess) { p->ty = nullptr; return MD2_ERR_CUDA; }
  for (int s = 1; s < p->num_scales; ++s)
    if (!p->level[s] &&
        md2_resize_plan_create(p->height >> (s - 1), p->width >> (s - 1), p->height >> s, p->width >> s, &p->level[s]) != MD2_OK)
      return MD2_ERR_CUDA;
  const int i = p->n_sizes;
  AxisTable ax, ay;
  bool ok = make_axis(w, p->width, &ax) && make_axis(h, p->height, &ay);
  if (ok) {
    const Table tx = as_table(ax), ty = as_table(ay);
    ok = cudaMemcpy(p->tx + i, &tx, sizeof(Table), cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(p->ty + i, &ty, sizeof(Table), cudaMemcpyHostToDevice) == cudaSuccess;
  }
  if (!ok) {
    free_axis(&ax); free_axis(&ay);
    return MD2_ERR_CUDA;
  }
  p->ax[i] = ax; p->ay[i] = ay;
  p->size_h[i] = h; p->size_w[i] = w;
  if (h > p->max_h) p->max_h = h;
  p->n_sizes = i + 1;
  *index = i;
  return MD2_OK;
}

int md2_batch_scratch_bytes(const md2_batch_plan* p, int n_images, int color_f32, size_t* bytes) {
  if (!p || !bytes || n_images < 1) return MD2_ERR_INVALID_ARGUMENT;
  *bytes = batch_scratch(p, n_images, color_f32).total;
  return MD2_OK;
}

int md2_batch_build_u8(const md2_batch_plan* p, const unsigned char* frames, size_t frames_bytes, const md2_batch_job* jobs,
                       const md2_batch_job* jobs_dev, int n_images, const md2_color_jitter* params, int n_samples,
                       void* out_color, int color_f32, float* out_color_aug, void* scratch, size_t scratch_bytes,
                       void* stream) {
  if (!p || !frames || !jobs || !jobs_dev || !params || !out_color || !out_color_aug || n_images < 1 || n_samples < 1)
    return MD2_ERR_INVALID_ARGUMENT;
  if ((long long)n_images * p->num_scales > 65535) return MD2_ERR_UNSUPPORTED;
  for (int i = 0; i < n_images; ++i) {
    const md2_batch_job& j = jobs[i];
    if (j.size < 0 || j.size >= p->n_sizes || p->size_h[j.size] != j.height || p->size_w[j.size] != j.width)
      return MD2_ERR_INVALID_ARGUMENT;                 // a size the plan does not hold
    if (j.offset < 0 || (size_t)j.offset > frames_bytes || frames_bytes - (size_t)j.offset < (size_t)3 * j.height * j.width)
      return MD2_ERR_INVALID_ARGUMENT;                 // would read outside `frames`
    if (j.sample < 0 || j.sample >= n_samples) return MD2_ERR_INVALID_ARGUMENT;
  }
  const BatchScratch sc = batch_scratch(p, n_images, color_f32);
  if (!scratch || scratch_bytes < sc.total) return MD2_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t s = (cudaStream_t)stream;
  const int n = n_images, H = p->height, W = p->width, S = p->num_scales;
  unsigned long long* sums = (unsigned long long*)scratch;
  unsigned char* tmp = (unsigned char*)scratch + sc.sums;
  unsigned char* lv = color_f32 ? tmp + sc.tmp : (unsigned char*)out_color;   // the uint8 levels
  CjImages im = {};
  im.n_img = n; im.n_levels = S;
  long long off = 0;
  for (int l = 0; l < S; ++l) {
    im.plane[l] = (H >> l) * (W >> l);
    im.off[l] = off;
    off += 3LL * n * im.plane[l];
  }
  // level 0 from the ragged, flipped native frames: every image in one launch per pass
  long long cnt = (long long)n * p->max_h * W;
  md2_resample_u8<0><<<(unsigned)((cnt + 255) / 256), 256, 0, s>>>(frames, tmp, jobs_dev, p->tx, n, 0, 0, p->max_h, W, 0,
                                                                    1, 1);
  cnt = (long long)n * H * W;
  md2_resample_u8<1><<<(unsigned)((cnt + 255) / 256), 256, 0, s>>>(tmp, lv, jobs_dev, p->ty, n, 0, W, H, W,
                                                                    3LL * p->max_h * W, 1, 0);
  // level l from level l-1 (mono_dataset.py:98-103), all images at once
  for (int l = 1; l < S; ++l) {
    const int st = md2_resize_lanczos_u8(p->level[l], lv + im.off[l - 1], lv + im.off[l], tmp, sc.tmp, n, 0, stream);
    if (st != MD2_OK) return st;
  }
  if (cudaMemsetAsync(sums, 0, (size_t)n * S * sizeof(unsigned long long), s) != cudaSuccess) return MD2_ERR_CUDA;
  cj_launch(lv, nullptr, out_color_aug, color_f32 ? (float*)out_color : nullptr, params, jobs_dev, sums, im, 0, s);
  return cudaGetLastError() == cudaSuccess ? MD2_OK : MD2_ERR_CUDA;
}

}  // extern "C"
