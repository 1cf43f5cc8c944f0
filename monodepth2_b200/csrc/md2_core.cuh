// md2_core.cuh - per-lane building blocks of the fused view-synthesis loss.
//
// Everything here is written as host/device functions of ONE lane's state so that
// the identical arithmetic runs (a) inside the sm_100a kernels of md2_kernels.cu, one
// lane per CUDA thread with warp shuffles between the stages, and (b) inside the
// lock-step host emulator of tests/emu (32 lanes in an array), which lets the tile /
// halo / reflection logic be checked against the oracle without a GPU.  The emulator
// is test infrastructure; the product path is the CUDA build only.
//
// Algorithm (reference file:line under /root/reference, restated per pixel in
// SURVEY.md Appendix A):
//   disp_s --bilinear up (trainer.py:350)--> D --(layers.py:16-25)--> depth z
//   cam = z * inv_K3 (x,y,1)          (layers.py:163-168)
//   cc  = (K T)[:3] (cam,1), u=cc0/(cc2+eps), v=cc1/(cc2+eps)   (layers.py:182-193)
//   border-clamped bilinear gather of the source at (u,v)        (trainer.py:384-387)
//   0.85*SSIM_3x3_reflect + 0.15*L1                              (trainer.py:393-405, layers.py:218-248)
//   per-pixel min over [identity+1e-5*noise, reprojection]       (trainer.py:426-484)
// and its adjoint back to D (then disp_s) and to the 3x4 projection P (then cam_T_cam).
#pragma once

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define MD2_HD __host__ __device__ __forceinline__
#else
#define MD2_HD inline
#endif

#if defined(__CUDA_ARCH__)
#define MD2_LD(p) __ldg(p)
#define MD2_LD4(p) __ldg(reinterpret_cast<const float4*>(p))
// streaming loads (read once per job: target row, disparity, identity loss, noise): do not allocate in
// L1, which is kept for the data-dependent gathers
#define MD2_LDS1(p) md2::ld_stream(p)
#define MD2_LDS4(p) md2::ld_stream4(p)
#define MD2_FMUL(a, b) __fmul_rn(a, b)
#define MD2_FADD(a, b) __fadd_rn(a, b)
#define MD2_RCP(a) md2::rcp_nr(a)
// the SSIM ratio n/d tolerates the 1-ulp MUFU.RCP result (loss parity budget 1e-5); the depth and
// projection reciprocals keep the Newton step because they decide bilinear cells
#define MD2_RCP_SSIM(a) md2::rcp_approx(a)
#define MD2_DIV(a, b) __fdiv_rn(a, b)
#define MD2_FLOORF(a) floorf(a)
#else
#define MD2_LD(p) (*(p))
#define MD2_LD4(p) (*reinterpret_cast<const md2::F4*>(p))
#define MD2_LDS1(p) (*(p))
#define MD2_LDS4(p) (*reinterpret_cast<const md2::F4*>(p))
#define MD2_FMUL(a, b) md2::host_fmul(a, b)
#define MD2_FADD(a, b) md2::host_fadd(a, b)
#define MD2_RCP(a) (1.0f / (a))
#define MD2_RCP_SSIM(a) (1.0f / (a))
#define MD2_DIV(a, b) ((a) / (b))
#define MD2_FLOORF(a) floorf(a)
#endif

namespace md2 {

#if defined(__CUDACC__)
typedef float4 F4;
#else
struct alignas(16) F4 { float x, y, z, w; };
#endif
MD2_HD F4 make_f4(float a, float b, float c, float d) { F4 r; r.x = a; r.y = b; r.z = c; r.w = d; return r; }

#if defined(__CUDA_ARCH__)
// MUFU.RCP + one Newton step: <= 1 ulp, 3 instructions instead of the IEEE sequence
__device__ __forceinline__ float ld_stream(const float* p) {
  float r;
  asm("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ F4 ld_stream4(const float* p) {
  F4 r;
  asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ float rcp_approx(float a) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
  return r;
}
__device__ __forceinline__ float rcp_nr(float a) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
  return fmaf(r, fmaf(-a, r, 1.0f), r);
}
#endif

#if defined(__CUDACC__)
// mbarrier + TMA bulk copy (cp.async.bulk, UBLKCP in SASS): global -> shared, completion by transaction bytes
__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* smem_dst, const void* gmem_src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_addr(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  unsigned done = 0;
  while (!done) {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(done) : "r"(smem_addr(bar)), "r"(parity) : "memory");
  }
}
#endif

#if !defined(__CUDA_ARCH__)
// keep the host compiler from contracting these into an fma
inline float host_fmul(float a, float b) { volatile float r = a * b; return r; }
inline float host_fadd(float a, float b) { volatile float r = a + b; return r; }
#endif

// Export of the discrete decisions the kernels take (bilinear cell + clip masks, per-pixel winner, SSIM
// clamp-live bits, L1 / smoothness signs) for the decision-locked fp64 test (SURVEY.md 8c, protocol P4).
// Two builds have it: the host emulator (g++), and the debug build of the CUDA library
// (-DMD2_DBG_DEVICE, libmd2loss_dbg.so, tests only); the product library compiles MD2_DBG to nothing.
struct DebugSink {
  int B, H, W, S, nsrc;
  short* x0;            // [S][B][nsrc][H][W]
  short* y0;
  unsigned char* mxy;   // bit0 = mx, bit1 = my
  signed char* tag;     // [S][B][H][W]   winner (-1: an identity candidate)
  unsigned char* live;  // [S][B][nsrc][3][H][W]  clamp-live bit of the SSIM window of source f, channel c
  signed char* l1sgn;   // [S][B][nsrc][3][H][W]  sign(pred - target)
  signed char* smx;     // per scale [B][Hs][Ws]  sign(n(p) - n(p+1x))
  signed char* smy;
  long smoff[4];
};
#if !defined(__CUDACC__)
inline DebugSink*& debug_sink() { static DebugSink* g = nullptr; return g; }
#define MD2_DBG_ON 1
#define MD2_DBG(...) do { if (md2::debug_sink()) { md2::DebugSink& D = *md2::debug_sink(); __VA_ARGS__; } } while (0)
#elif defined(MD2_DBG_DEVICE)
static __device__ DebugSink g_dbg_sink;      // all-null = off; set by md2_debug_set_sink (md2_kernels.cu)
#define MD2_DBG_ON 1
#if defined(__CUDA_ARCH__)
#define MD2_DBG(...) do { if (md2::g_dbg_sink.x0) { md2::DebugSink& D = md2::g_dbg_sink; __VA_ARGS__; } } while (0)
#else
#define MD2_DBG(...) do { } while (0)
#endif
#else
#define MD2_DBG_ON 0
#define MD2_DBG(...) do { } while (0)
#endif

// Debug build only (-DMD2_BOUNDS_CHECK): every index the marching path uses for a global load / store is
// checked against the extent of its tensor; violations are counted (md2_debug_oob_count), the access is skipped
// by clamping.  compute-sanitizer is closed on the pool this was developed on; this is its stand-in.
#if defined(MD2_BOUNDS_CHECK) && defined(__CUDACC__)
static __device__ unsigned long long g_oob_count;
#endif
#if defined(MD2_BOUNDS_CHECK) && defined(__CUDA_ARCH__)
#define MD2_CHK(idx, n) do { if ((unsigned)(idx) >= (unsigned)(n)) atomicAdd(&md2::g_oob_count, 1ULL); } while (0)
#else
#define MD2_CHK(idx, n) do { } while (0)
#endif

constexpr int kMaxScales = 4;
constexpr int kMaxSrc = 4;
constexpr int kLanes = 32;
constexpr int kOwnCols = 28;   // columns a marching warp owns (32 lanes - 2x2 halo)
constexpr int kIdCols = 30;    // columns the identity pass owns (32 lanes - 2x1 halo)
constexpr int kRing = 3;       // rows kept in the per-thread stash ring

constexpr float kSsimC1 = 0.0001f;
constexpr float kSsimC2 = 0.0009f;

// Device-side view of one evaluation (filled by the host planner in md2_plan.h).
struct Params {
  int B, H, W, S, nsrc, nid;
  int automask, avg, align_corners, want_grad, no_ssim;
  // --pose_model_type posecnn (trainer.py:366-375): one T per (scale, sample, source), built from the pose leaves
  // with the translation multiplied by the mean inverse depth of the scale.  npose = S (posecnn) or 1: the number of
  // projection tables / pose-gradient accumulators per (sample, source).
  int posecnn, npose;
  // --predictive_mask (trainer.py:447-459)
  int pmask_on;
  float a_disp, c_disp;      // scaled_disp = a + c*disp            layers.py:21-23
  float sx, ox, sy, oy;      // ix = u*sx + ox ; iy = v*sy + oy     (grid normalise o unnormalise)
  float wmax, hmax;          // W-1, H-1
  float eps;
  float gscale;              // 1/(S*B*H*W) [* 1/nsrc under avg_reprojection]
  float smooth_w[kMaxScales];  // disparity_smoothness / 2^lvl[s]
  int seg_rows, nseg, nband, nband_id;
  int nsm;                   // SMs of the device (role rotation of the role-specialised kernel)
  int id_rows, nseg_id;      // row segments of the (much lighter) identity pass
  const float* tgt;
  const float* src[kMaxSrc];
  const float* Tm[kMaxSrc];
  int pose_grad[kMaxSrc];
  // pose leaves (optional, per source): when aa[f] is set the call builds T_f itself (SURVEY.md 8f rank 1)
  const float* aa[kMaxSrc];        // axisangle, 3 floats per sample, `pose_stride[f]` floats between samples
  const float* tr[kMaxSrc];        // translation, same layout
  int pose_stride[kMaxSrc];
  int pose_invert[kMaxSrc];        // frame_id < 0 (trainer.py:294-295)
  float* Tws[kMaxSrc];             // (B,4,4) workspace / output: the T built from the leaves
  float* grad_aa[kMaxSrc];         // (B,3) d loss / d axisangle
  float* grad_tr[kMaxSrc];         // (B,3) d loss / d translation
  // uint8 image inputs (optional, md2_tensors::target_u8 ...): what the dataloader holds before ToTensor
  // (datasets/mono_dataset.py:106-109); converted with x / 255 (IEEE division = torchvision's ToTensor) where
  // the float images would have been read.  u8_hwc: (B,H,W,3) interleaved, else (B,3,H,W) planar.
  const unsigned char* tgt8;
  const unsigned char* src8[kMaxSrc];
  const unsigned char* color8[kMaxScales];
  int u8_hwc;
  const float* K;
  const float* invK;
  const float* disp[kMaxScales];
  const float* color[kMaxScales];
  const float* noise[kMaxScales];
  void* noise_event;               // host side only: cudaEvent_t the marching kernel's launch waits for (md2_tensors.noise_ready_event)
  // workspace
  float* tgt4;             // (B,H,W,4) target re-laid out as RGBx texels
  float* src4[kMaxSrc];    // (B,H,W,4) sources as RGBx texels: one 16-byte load per bilinear tap
  float* proj;     // (B,nsrc,12): M=P3*invK3 (row-major 3x3) then p4
  float* idloss;   // (B,nsrc,H,W)
  float* dD[kMaxScales];   // (B,H,W)   d loss / d upsampled disp_s
  float* zup[kMaxScales];  // (B,H,W)   depth of the up-sampled disp_s (md2_depth_up; read by role A of the role kernels)
  float* gn[kMaxScales];   // (B,Hs,Ws) smoothness numerator gradient
  float* smsc;             // (S,B,2): 1/m and (sum gn*disp)/(m^2 N) of the smoothness adjoint, as floats
  float* mid;              // posecnn: (S,B) mean inverse depth of the up-sampled disparity (trainer.py:371-372)
  float* gmidc;            // posecnn: (S,B) d loss / d (every pixel of the up-sampled disp_s) through mean_inv_depth
  // uint8 entry: the frames (and the target pyramid) converted once to planar float, so that every later pass runs
  // its float form (the TMA-staged identity pass reads planar float through tensor maps)
  float* cvt_img[1 + kMaxSrc];      // (B,3,H,W): target, sources
  float* cvt_col[kMaxScales];       // (B,3,Hs,Ws), s >= 1
  const float* pmask[kMaxScales];   // predictive mask, (B,nsrc,Hs,Ws)
  float* pm[kMaxScales];            // (B,nsrc,H,W) mask up-sampled to full resolution (trainer.py:451-454)
  float* gpm[kMaxScales];           // (B,nsrc,H,W) d loss / d up-sampled mask (photometric part)
  float* grad_pmask[kMaxScales];    // out (B,nsrc,Hs,Ws)
  double* acc;     // accumulators, layout below
  // outputs
  float* losses;
  float* grad_disp[kMaxScales];
  float* grad_T[kMaxSrc];
  float* depth[kMaxScales];
  float* warped[kMaxSrc][kMaxScales];
  float* idsel[kMaxScales];
  // --scales subsets (options.py:64).  At the end of the struct: the constant-bank offsets of every field above are
  // the ones the marching kernels were tuned with.
  int lvl[kMaxScales];         // pyramid level of scale slot s: opt.scales sorted ascending (trainer.py:345,413); slot s holds
                               // (H >> lvl[s], W >> lvl[s]) tensors.  0..S-1 for the default --scales 0 1 2 3.  lvl[0] == 0
                               // always (validate(): the reference needs level 0, trainer.py:377), so "slot 0" and
                               // "full resolution, no up-sampling" are the same thing in every kernel
  int up0;                     // first slot that is up-sampled (= 1)
  int lvl4;                    // the same levels, 4 bits per slot: level of slot s = (lvl4 >> 4 s) & 15 (make_job: plain shifts
                               // of one kernel parameter instead of an indexed constant load - same code as `>> s` had)
};

// accumulator layout (doubles)
MD2_HD int acc_photo(int s) { return s; }
// (slots [kMaxScales, 3 kMaxScales) are unused: the smoothness sums are kept per (scale, sample), see
// acc_smx / acc_smy below, so that the blocks of md2_smooth do not all hit two addresses per scale)
MD2_HD int acc_dispsum(const Params& P, int s, int b) { return 3 * kMaxScales + s * P.B + b; }
MD2_HD int acc_dot(const Params& P, int s, int b) { return 3 * kMaxScales + kMaxScales * P.B + s * P.B + b; }
// ps: pose set (the scale under posecnn, else 0)
MD2_HD int acc_dP(const Params& P, int ps, int b, int f, int k) {
  return 3 * kMaxScales + 2 * kMaxScales * P.B + ((ps * P.B + b) * P.nsrc + f) * 12 + k;
}
MD2_HD int acc_smx(const Params& P, int s, int b) {
  return 3 * kMaxScales + 2 * kMaxScales * P.B + P.npose * P.B * P.nsrc * 12 + 2 * (s * P.B + b);
}
MD2_HD int acc_smy(const Params& P, int s, int b) { return acc_smx(P, s, b) + 1; }
// posecnn: sum of the up-sampled disparity of (scale, sample) over the full-resolution grid
MD2_HD int acc_updisp(const Params& P, int s, int b) {
  return 3 * kMaxScales + 4 * kMaxScales * P.B + P.npose * P.B * P.nsrc * 12 + s * P.B + b;
}
// predictive mask: sum of -log(mask) over the up-sampled mask of scale s (BCE against ones, trainer.py:458)
MD2_HD int acc_bce(const Params& P, int s) {
  return 3 * kMaxScales + 5 * kMaxScales * P.B + P.npose * P.B * P.nsrc * 12 + s;
}
MD2_HD int acc_count(const Params& P) {
  return 3 * kMaxScales + 5 * kMaxScales * P.B + P.npose * P.B * P.nsrc * 12 + kMaxScales;
}

// ToTensor (torchvision.transforms.functional.to_tensor): uint8 -> float32, then .div(255)
// Device: q = v * rn(1/255) followed by one Newton correction, rem = fma(-q, 255, v), q' = fma(rem, rn(1/255), q), is
// the correctly rounded quotient for every one of the 256 byte values (checked exhaustively against the IEEE division,
// tests/test_u8_entry.py) - three instructions instead of the division's slow path, nine times per pixel and row.
MD2_HD float u8_unit(unsigned char v) {
#if defined(__CUDA_ARCH__)
  const float x = (float)v, r = 0.003921568859368563f;      // rn(1 / 255)
  const float q = x * r;
  return fmaf(fmaf(-q, 255.0f, x), r, q);
#else
  return MD2_DIV((float)v, 255.0f);
#endif
}
// channel c of pixel `pix` (= y * w + x) of sample b of a 3-channel image given as float planar NCHW (`f32`)
// or, when `u8` is set, as uint8 (planar or interleaved); `plane` = h * w of that image
MD2_HD float load_px(const float* f32, const unsigned char* u8, int hwc, int b, int c, int plane, int pix) {
  if (u8) {
    const size_t o = hwc ? ((size_t)b * plane + pix) * 3 + c : ((size_t)b * 3 + c) * plane + pix;
#if defined(__CUDA_ARCH__)
    return u8_unit(__ldg(u8 + o));
#else
    return u8_unit(u8[o]);
#endif
  }
  return MD2_LD(f32 + ((size_t)b * 3 + c) * plane + pix);
}

// One marching job (warp-uniform): a band of kOwnCols columns x rows [y0,y1) of sample b at
// scale s, with every base pointer already offset to the sample so that per-pixel addressing
// is 32-bit index arithmetic (validate() bounds the tensors below 2^31 elements).
struct WarpJob {
  int s, b;
  // (slot s is at full resolution - level 0, no up-sampling - iff s == 0: validate() requires level 0 in the list)
  int ps;        // pose set: s under posecnn, else 0
  const float* proj;   // projection table of (ps, b): nsrc x 12 floats
  const float* pm;     // predictive mask up-sampled to (H,W), planes [nsrc] of sample b at scale s (or null)
  float* gpm;          // its gradient planes (or null)
  int x0;        // first owned column
  int y0, y1;    // owned rows [y0, y1)
  int H, W, Hs, Ws, plane;
  float rs;      // 1 / 2^s
  const float* tgt4;
  const float* src4[kMaxSrc];
  const float* disp;
  const float* zup;    // depth plane of (s, b) at full resolution (Cfg::ZUP)
  const float* idl;
  const float* noise;
  float* dD;
  // scale 0 only: the smoothness adjoint is added in place and grad_disp_0 written directly
  float* gd0;
  const float* gn0;
  float sm_inv_m, sm_dterm, sm_w;
  float* idsel;
  float* depth;
  float* warped[kMaxSrc];
  // role-specialised kernel, interior bands: the target texel row is put into the ring by a TMA bulk copy
  // (field 0 of the slot = 32 consecutive RGBx texels) instead of being loaded and stored by every lane
  int staged;
};

MD2_HD void smooth_scalars(const Params& P, int s, int b, float& inv_m, float& dterm);

MD2_HD WarpJob make_job(const Params& P, int s, int b, int x0, int y0, int y1) {
  WarpJob J;
  const int lv = (P.lvl4 >> (4 * s)) & 15;
  J.s = s; J.b = b; J.x0 = x0; J.y0 = y0; J.y1 = y1;
  J.H = P.H; J.W = P.W; J.Hs = P.H >> lv; J.Ws = P.W >> lv; J.plane = P.H * P.W;
  J.rs = 1.0f / (float)(1 << lv);
  J.ps = P.posecnn ? s : 0;
  J.proj = P.proj + (size_t)((J.ps * P.B + b) * P.nsrc) * 12;
  const int boff = b * J.plane;
  J.pm = (P.pmask_on && P.pm[s]) ? P.pm[s] + (size_t)P.nsrc * boff : nullptr;
  J.gpm = (P.pmask_on && P.want_grad && P.gpm[s]) ? P.gpm[s] + (size_t)P.nsrc * boff : nullptr;
  J.tgt4 = P.tgt4 + 4 * boff;
  for (int f = 0; f < kMaxSrc; ++f) {
    J.src4[f] = f < P.nsrc ? P.src4[f] + 4 * boff : nullptr;
    J.warped[f] = (f < P.nsrc && P.warped[f][s]) ? P.warped[f][s] + 3 * boff : nullptr;
  }
  J.disp = P.disp[s] + b * J.Hs * J.Ws;
  // (scale 0 needs no up-sampling: the plane is the disparity itself, turned into depth by the reader)
  J.zup = s == 0 ? J.disp : (P.zup[s] ? P.zup[s] + boff : nullptr);
  J.idl = P.idloss + P.nsrc * boff;
  J.noise = P.noise[s] ? P.noise[s] + P.nid * boff : nullptr;
  J.dD = P.dD[s] + boff;
  J.gd0 = nullptr; J.gn0 = nullptr; J.sm_inv_m = 0.f; J.sm_dterm = 0.f; J.sm_w = 0.f;
  if (s == 0 && P.want_grad) {
    J.gd0 = P.grad_disp[0] + boff;
    J.gn0 = P.gn[0] + boff;
    J.sm_inv_m = MD2_LD(P.smsc + 2 * b);            // scale 0, sample b
    J.sm_dterm = MD2_LD(P.smsc + 2 * b + 1);
    J.sm_w = P.smooth_w[0] / (float)P.S;
  }
  J.idsel = P.idsel[s] ? P.idsel[s] + boff : nullptr;
  J.depth = P.depth[s] ? P.depth[s] + boff : nullptr;
  J.staged = 0;
  return J;
}

template <int NSRC_, bool AVG_, bool AUTOMASK_, bool GRAD_, bool NOSSIM_ = false>
struct Cfg {
  static constexpr int NSRC = NSRC_;
  static constexpr bool NOSSIM = NOSSIM_;                        // --no_ssim: L1 only (trainer.py:399-400)
  static constexpr bool AVG = AVG_;
  static constexpr bool AUTOMASK = AUTOMASK_;
  static constexpr bool GRAD = GRAD_;
  static constexpr int NCS = AVG_ ? NSRC_ : 1;                   // coefficient sets shipped per window
  static constexpr int NID = AUTOMASK_ ? (AVG_ ? 1 : NSRC_) : 0; // identity candidates
  static constexpr int STASH4 = 1 + 3 * NSRC_;                   // 16-byte fields per ring row
  // ZUP: the depth of every full-resolution pixel of every scale comes from a plane written by md2_depth_up before the
  // marching kernel (one coalesced load per lane and row) instead of being rebuilt per row from four disparity taps,
  // the up-sampling weights and a reciprocal.  The role-specialised kernels set it (RoleOf): their role A is the role
  // every barrier waits for, and this takes ~45 instructions per row and the head of its dependent chain out of it.
  static constexpr bool ZUP = false;
  // PAIRED (packed two-source role kernel, md2_roles.cuh PairedOf): ring fields 1 and 4 hold (r0, g0, r1, g1) and
  // (b0, b1, u0, u1) - the aligned register pairs role B's f32x2 arithmetic reads - instead of (r, g, b, u) per source
  static constexpr bool PAIRED = false;
  // Backward rolling state (two rows of 9*NSRC box sums): registers for up to two sources, a
  // thread-private shared-memory ring beyond that (3 sources would spill ~0.5 KB per thread).
  static constexpr bool BSMEM = GRAD_ && (NSRC_ >= 3);
  // Control-flow shape of stages B/C: with 3 sources the branch-free form (every lane computes, results
  // masked) is 7 % faster, with 1-2 sources the divergent form is 3 % faster (measured, r01 log).
  static constexpr bool STRAIGHT = (NSRC_ >= 3);
  static constexpr int NB4 = (9 * NSRC_ + 3) / 4;                // 16-byte fields per B row
  static constexpr int SMEM4 = (GRAD_ ? kRing * STASH4 : 0) + (BSMEM ? 2 * NB4 : 0);  // per thread
};

// ------------------------------------------------------------------ SSIM pieces
// Sums over the 3x3 window: sx=Σx, sxx=Σx², sxy=Σxy, sy=Σy, syy=Σy².
// Returns clamp((1 - n/d)/2, 0, 1)  (layers.py:238-248).  The means and (co)variances are
// kept multiplied by 9 / 81 (the factors cancel in n/d), which avoids the 1/9 constant
// whose fp32 rounding would be amplified by the E[x^2]-mu^2 cancellation:
//   81 n1 = 2 sx sy + 81 C1          81 n2 = 2 (9 sxy - sx sy) + 81 C2
//   81 d1 = sx^2 + sy^2 + 81 C1      81 d2 = 9 (sxx + syy) - sx^2 - sy^2 + 81 C2
// When `coef` is non-null it receives -0.5*live*(alpha, beta, gamma) with
// d(n/d)/dx_j = alpha + beta*x_j + gamma*y_j for every x_j of the window (SURVEY.md A.2).
MD2_HD float ssim_window(float sx, float sxx, float sxy, float sy, float syy, float* coef, bool valid = true,
                         unsigned char* live_out = nullptr) {
  const float c1 = 81.0f * kSsimC1, c2 = 81.0f * kSsimC2;
  const float pxy = sx * sy;
  const float pp = fmaf(sx, sx, sy * sy);
  const float n1 = fmaf(2.0f, pxy, c1);
  const float n2 = fmaf(2.0f, fmaf(9.0f, sxy, -pxy), c2);
  const float d1 = pp + c1;
  const float d2 = fmaf(9.0f, sxx + syy, -pp) + c2;
  const float N = n1 * n2, D = d1 * d2;
  const float invD = MD2_RCP_SSIM(D);
  const float Q = N * invD;
  const float raw = fmaf(-0.5f, Q, 0.5f);
  const float S = fminf(fmaxf(raw, 0.0f), 1.0f);
  if (coef) {
    const bool live = (raw >= 0.0f) && (raw <= 1.0f);
    if (MD2_DBG_ON && live_out) *live_out = live ? 1 : 0;
    const float k = (live && valid) ? -0.5f : 0.0f;
    const float QD = Q * invD;                       // N / D^2
    const float alpha = 2.0f * (sy * (n2 - n1) * invD - sx * (d2 - d1) * QD);
    const float beta = -18.0f * d1 * QD;
    const float gamma = 18.0f * n1 * invD;
    coef[0] = k * alpha;
    coef[1] = k * beta;
    coef[2] = k * gamma;
  }
  return S;
}

// index reflection of ReflectionPad2d(1) (layers.py:235-236), then clamped so that lanes /
// rows beyond the pad ring still address valid memory (their values are never used)
MD2_HD int reflect_clamp(int i, int n) {
  i = i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i);
  return i < 0 ? 0 : (i >= n ? n - 1 : i);
}

// ------------------------------------------------------------------ lane state
// What stage_a_issue hands to stage_a_finish: the gather of one row in flight.
template <class C>
struct Flight {
  F4 tap[C::NSRC][4];                           // nw, ne, sw, se texels
  float cz;                                     // depth
  float cu[C::NSRC], cv[C::NSRC];               // projected pixel coordinates
  float cwx[C::NSRC], cwy[C::NSRC];             // bilinear weights
  float cgx[C::NSRC], cgy[C::NSRC];             // clip mask * d(ix,iy)/d(u,v) / den
  F4 ctg;                                       // target texel of the row
};

template <class C>
struct Lane {
  // constants of the job
  int x;            // column of this lane (may be outside the image)
  int xi;           // reflected/clamped column: where this lane actually reads
  bool colok;
  float qa[C::NSRC][3];   // M[i][0]*xi + M[i][2]
  float qb[C::NSRC][3];   // M[i][1]
  float p4[C::NSRC][3];   // (K T)[i][3]
  int ux0, ux1;           // bilinear up-sampling taps of disp_s in x
  float ul0, ul1;
  // software prefetch: inputs of the NEXT row, in flight during the current step
  F4 ntg;                 // target texel of row t+1
  float nd[4];            // disparity taps of row t+1 (d00,d01,d10,d11; scale 0: d00 only)
  // gather of the current row, in flight between stage_a_issue and stage_a_finish
  Flight<C> fl;
  // identity loss + noise of the current window row (loaded at the top of the step)
  float idv[C::NSRC], nzv[C::NSRC];
  // forward rolling state (horizontal 3-sums of the two previous rows)
  float H1[C::NSRC][3][3], H2[C::NSRC][3][3];   // [f][c][x,xx,xy]: previous row | sum of the two previous rows
  float HY1[3][2], HY2[3][2];                   // [c][y,yy]
  float pr1[C::NSRC][3], tg1[3];                // own pred / target of the previous row
  // exports of the current step
  float pr[C::NSRC][3], tg[3];
  float coef[C::NCS][9];                        // [set][c*3 + {alpha,beta,gamma}]
  int tag;                                      // winner of the current window row
  // backward rolling state
  float B1[C::NSRC][9], B2[C::NSRC][9];
  int tag1;                                     // winner one window row earlier
  // accumulators
  float loss;
  float S1[C::NSRC][3], S2[C::NSRC][3], S3[C::NSRC][3];
};

template <class C>
struct Xchg1 {   // what stage B needs from a horizontal neighbour
  float pr[C::NSRC][3];
  float tg[3];
};
template <class C>
struct Xchg2 {   // what stage C needs from a horizontal neighbour
  float coef[C::NCS][9];
  int tag;
};

MD2_HD int ring_slot(int t) { return ((t % kRing) + kRing) % kRing; }

// thread-private stash of 16-byte fields: element (slot, field) of this lane; consecutive
// lanes are 16 bytes apart, so 128-bit shared accesses are conflict-free
template <int R>
struct StashT {
  static constexpr int kDepth = R;   // rows kept in the ring
  F4* base;
  F4* bring;      // ring of 2 rows x NB4 fields (backward box sums), only when Cfg::BSMEM
  int stride;     // threads sharing the ring (lane stride of one field)
  unsigned long long* tbar;   // WarpJob::staged: one mbarrier per slot, armed by the TMA copy of the target row
  int t0;                     // first row of the job (the n-th use of a slot completes phase n of its mbarrier)
  MD2_HD int slot(int t) const { return ((t % R) + R) % R; }
  MD2_HD unsigned parity(int t) const { return (unsigned)(((t - t0) / R) & 1); }
  MD2_HD F4& at(int slot, int field, int nfields) const { return base[(slot * nfields + field) * stride]; }
  MD2_HD F4& b(int slot, int field, int nfields) const { return bring[(slot * nfields + field) * stride]; }
};
typedef StashT<kRing> Stash;

// one bilinear blend of the disparity up-sampling, w0 a + w1 b, with the contraction spelled out: the same bits in
// every kernel that up-samples (marching kernels, md2_depth_up) and in the host emulator, whatever the compiler would
// have fused on its own
MD2_HD float up_blend(float w0, float a, float w1, float b) { return fmaf(w1, b, MD2_FMUL(w0, a)); }

// layers.py:16-25: depth = 1 / (min_disp + (max_disp - min_disp) * disp)
MD2_HD float depth_of_disp(const Params& P, float D) {
  const float sd = MD2_FADD(P.a_disp, MD2_FMUL(P.c_disp, D));
  return MD2_RCP(sd);
}

// issue the loads of row `t`'s target texel and disparity taps (consumed one step later)
template <class C, bool WITH_TG = true>
MD2_HD void prefetch_row(Lane<C>& L, const WarpJob& J, int t) {
  const int tr = reflect_clamp(t, J.H);
  MD2_CHK(tr * J.W + L.xi, J.plane);
  if (WITH_TG) L.ntg = MD2_LDS4(J.tgt4 + 4 * (tr * J.W + L.xi));
  if (C::ZUP) {
    L.nd[0] = MD2_LD(J.zup + tr * J.W + L.xi);
  } else if (J.s == 0) {
    L.nd[0] = MD2_LD(J.disp + tr * J.W + L.xi);
  } else {
    float syr = fmaf(J.rs, (float)tr + 0.5f, -0.5f);
    syr = syr < 0.0f ? 0.0f : syr;
    const int y0 = (int)syr;
    const int y1 = y0 + ((y0 < J.Hs - 1) ? 1 : 0);
    const float* r0 = J.disp + y0 * J.Ws;
    const float* r1 = J.disp + y1 * J.Ws;
    MD2_CHK(y0 * J.Ws + L.ux0, J.Hs * J.Ws); MD2_CHK(y1 * J.Ws + L.ux1, J.Hs * J.Ws);
    L.nd[0] = MD2_LD(r0 + L.ux0); L.nd[1] = MD2_LD(r0 + L.ux1);
    L.nd[2] = MD2_LD(r1 + L.ux0); L.nd[3] = MD2_LD(r1 + L.ux1);
  }
}

template <class C>
MD2_HD void lane_init(Lane<C>& L, const Params& P, const WarpJob& J, int lane) {
  L.x = J.x0 - 2 + lane;
  L.colok = (L.x >= 0) && (L.x < P.W);
  L.xi = reflect_clamp(L.x, P.W);
  const float xf = (float)L.xi;
#pragma unroll
  for (int f = 0; f < C::NSRC; ++f) {
    const float* m = J.proj + f * 12;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      L.qa[f][i] = fmaf(MD2_LD(m + i * 3 + 0), xf, MD2_LD(m + i * 3 + 2));
      L.qb[f][i] = MD2_LD(m + i * 3 + 1);
      L.p4[f][i] = MD2_LD(m + 9 + i);
    }
    L.idv[f] = 0.f; L.nzv[f] = 0.f;
  }
  if (J.s > 0) {
    float sxr = fmaf(J.rs, (float)L.xi + 0.5f, -0.5f);
    sxr = sxr < 0.0f ? 0.0f : sxr;
    L.ux0 = (int)sxr;
    L.ux1 = L.ux0 + ((L.ux0 < J.Ws - 1) ? 1 : 0);
    L.ul1 = sxr - (float)L.ux0;
    L.ul0 = 1.0f - L.ul1;
  } else {
    L.ux0 = L.ux1 = L.xi;
    L.ul0 = 1.0f; L.ul1 = 0.0f;
  }
  L.nd[0] = L.nd[1] = L.nd[2] = L.nd[3] = 0.f;
#pragma unroll
  for (int f = 0; f < C::NSRC; ++f) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
      for (int k = 0; k < 3; ++k) { L.H1[f][c][k] = 0.f; L.H2[f][c][k] = 0.f; }
      L.pr1[f][c] = 0.f; L.pr[f][c] = 0.f;
      L.S1[f][c] = 0.f; L.S2[f][c] = 0.f; L.S3[f][c] = 0.f;
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) { L.B1[f][k] = 0.f; L.B2[f][k] = 0.f; }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    L.HY1[c][0] = L.HY1[c][1] = L.HY2[c][0] = L.HY2[c][1] = 0.f;
    L.tg1[c] = 0.f; L.tg[c] = 0.f;
  }
#pragma unroll
  for (int n = 0; n < C::NCS; ++n)
#pragma unroll
    for (int k = 0; k < 9; ++k) L.coef[n][k] = 0.f;
  L.tag = -1; L.tag1 = -1;
  L.loss = 0.f;
  prefetch_row(L, J, J.y0 - 2);
}

// zero the shared-memory ring of backward box sums at the start of a job
template <class C, class ST>
MD2_HD void bring_reset(const ST& st) {
  if (C::BSMEM) {
#pragma unroll
    for (int i = 0; i < 2 * C::NB4; ++i) st.bring[i * st.stride] = make_f4(0.f, 0.f, 0.f, 0.f);
  }
}

// ------------------------------------------------------------------ stage A
// Row t is read at its reflected position, so pad-ring rows/lanes carry the reflected values
// and no edge case is needed downstream.
// stage_a_issue: up-sampled disparity (trainer.py:350-351, torch upsample_bilinear2d,
// align_corners=False) -> depth (layers.py:16-25) -> projection into every source
// (layers.py:139-193) -> border-clamped bilinear cell (trainer.py:384-387); issues the 4 tap
// loads per source and the loads of the following row (target, disparity) and of the identity
// loss / noise of window row t-1.  Nothing here waits for memory: the caller runs the adjoint of
// an earlier row (stage_c) while the gather is in flight.
// identity loss + tie-break noise of window row t-1 (consumed by stage_b of step t)
template <class C>
MD2_HD void load_identity_row(Lane<C>& L, const WarpJob& J, int t) {
  if (C::AUTOMASK) {
    const int yw = t - 1;
    const int pix = (yw < 0 ? 0 : (yw >= J.H ? J.H - 1 : yw)) * J.W + L.xi;
    MD2_CHK(pix, J.plane);
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f) L.idv[f] = MD2_LDS1(J.idl + f * J.plane + pix);
#pragma unroll
    for (int f = 0; f < C::NID; ++f) L.nzv[f] = MD2_LDS1(J.noise + f * J.plane + pix);
  } else if (J.pm) {
    // --predictive_mask (needs --disable_automasking, trainer.py:90-92): the up-sampled mask of window row t-1
    const int yw = t - 1;
    const int pix = (yw < 0 ? 0 : (yw >= J.H ? J.H - 1 : yw)) * J.W + L.xi;
    MD2_CHK(pix, J.plane);
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f) L.nzv[f] = MD2_LDS1(J.pm + f * J.plane + pix);
  }
}

// --predictive_mask, stage B (trainer.py:456): reprojection_losses *= mask, before the mean / minimum over sources.
// rl keeps the unmasked loss (it is d loss / d mask of the winner), rlm receives the masked one.
template <class C>
MD2_HD void pmask_apply(const Lane<C>& L, const WarpJob& J, const float* rl, float* rlm) {
#pragma unroll
  for (int f = 0; f < C::NSRC; ++f) rlm[f] = (!C::AUTOMASK && J.pm) ? rl[f] * L.nzv[f] : rl[f];
}
// d loss / d (up-sampled mask) of the window pixel (photometric part; the BCE part is added by the final pass),
// and the winner's SSIM-adjoint coefficients scaled by its mask value
template <class C>
MD2_HD void pmask_backward(Lane<C>& L, const Params& P, const WarpJob& J, const float* rl, int tag, bool own_win, int yw) {
  if (C::AUTOMASK || !J.pm) return;
  if (C::GRAD) {
#pragma unroll
    for (int n = 0; n < C::NCS; ++n) {
      float m = L.nzv[0];
      if (C::AVG) m = L.nzv[n];
      else {
#pragma unroll
        for (int f = 1; f < C::NSRC; ++f) m = (tag == f) ? L.nzv[f] : m;
      }
#pragma unroll
      for (int k = 0; k < 9; ++k) L.coef[n][k] *= m;
    }
    if (own_win && J.gpm) {
#pragma unroll
      for (int f = 0; f < C::NSRC; ++f)
        J.gpm[f * J.plane + yw * J.W + L.xi] = (C::AVG ? (tag >= 0) : (tag == f)) ? rl[f] * P.gscale : 0.0f;
    }
  }
}

// ROW_STEP: distance to the row this warp handles next (its target / disparity loads are put in flight here)
// TG_DIRECT: the target texel of row t is loaded here, straight into the slot stage_a_finish reads (it is not
// needed before), instead of being prefetched one step ahead and moved: a move placed after the gather issue
// waits on the gather's scoreboard (role kernel, measured: 10 % of all stall samples on that one MOV)
template <class C, bool WITH_ID = true, int ROW_STEP = 1, bool TG_DIRECT = false>
MD2_HD void stage_a_issue(Lane<C>& L, Flight<C>& F, const Params& P, const WarpJob& J, int t) {
  const int tr = reflect_clamp(t, J.H);
  MD2_CHK(tr * J.W + L.xi, J.plane);
  if (TG_DIRECT) {
    if (J.staged) F.ctg = make_f4(0.f, 0.f, 0.f, 0.f);      // the row goes into the ring by TMA
    else F.ctg = MD2_LDS4(J.tgt4 + 4 * (tr * J.W + L.xi));
  } else F.ctg = L.ntg;
  float D = 0.f, zpre = 0.f;
  if (C::ZUP) {
    zpre = L.nd[0];
  } else if (J.s == 0) {
    D = L.nd[0];
  } else {
    float syr = fmaf(J.rs, (float)tr + 0.5f, -0.5f);
    syr = syr < 0.0f ? 0.0f : syr;
    const float l1 = syr - (float)(int)syr, l0 = 1.0f - l1;
    const float top = up_blend(L.ul0, L.nd[0], L.ul1, L.nd[1]);
    const float bot = up_blend(L.ul0, L.nd[2], L.ul1, L.nd[3]);
    D = up_blend(l0, top, l1, bot);
  }
  if (ROW_STEP > 0) prefetch_row<C, !TG_DIRECT>(L, J, t + ROW_STEP);     // ROW_STEP 0: the caller prefetches
  if (WITH_ID) load_identity_row(L, J, t);
  const float z = C::ZUP ? (J.s == 0 ? depth_of_disp(P, zpre) : zpre) : depth_of_disp(P, D);
  F.cz = z;
  const float yf = (float)tr;
#pragma unroll
  for (int f = 0; f < C::NSRC; ++f) {
    const float q0 = fmaf(L.qb[f][0], yf, L.qa[f][0]);
    const float q1 = fmaf(L.qb[f][1], yf, L.qa[f][1]);
    const float q2 = fmaf(L.qb[f][2], yf, L.qa[f][2]);
    const float c0 = fmaf(z, q0, L.p4[f][0]);
    const float c1 = fmaf(z, q1, L.p4[f][1]);
    const float c2 = fmaf(z, q2, L.p4[f][2]);
    const float inv = MD2_RCP(c2 + P.eps);
    const float u = c0 * inv;
    const float v = c1 * inv;
    const float ix = fmaf(u, P.sx, P.ox);
    const float iy = fmaf(v, P.sy, P.oy);
    const bool mx = (ix > 0.0f) && (ix < P.wmax);
    const bool my = (iy > 0.0f) && (iy < P.hmax);
    const float ixc = fminf(fmaxf(ix, 0.0f), P.wmax);
    const float iyc = fminf(fmaxf(iy, 0.0f), P.hmax);
    const float fx0 = MD2_FLOORF(ixc), fy0 = MD2_FLOORF(iyc);
    const int x0 = (int)fx0, y0 = (int)fy0;
    MD2_DBG(if (L.colok && t >= 0 && t < J.H) {
      const long o = ((((long)J.s * D.B + J.b) * D.nsrc + f) * D.H + t) * D.W + L.x;
      D.x0[o] = (short)x0; D.y0[o] = (short)y0; D.mxy[o] = (unsigned char)((mx ? 1 : 0) | (my ? 2 : 0));
    });
    const int dx1 = (x0 + 1 < J.W) ? 4 : 0;                 // texel step to the east tap
    const int dy1 = (y0 + 1 < J.H) ? J.W * 4 : 0;           // texel step to the south tap
    const float* t00 = J.src4[f] + 4 * (y0 * J.W + x0);
    MD2_CHK(y0 * J.W + x0, J.plane); MD2_CHK(y0 * J.W + x0 + (dx1 + dy1) / 4, J.plane);
    F.tap[f][0] = MD2_LD4(t00);
    F.tap[f][1] = MD2_LD4(t00 + dx1);
    F.tap[f][2] = MD2_LD4(t00 + dy1);
    F.tap[f][3] = MD2_LD4(t00 + dy1 + dx1);
    F.cu[f] = u; F.cv[f] = v;
    F.cwx[f] = ixc - fx0; F.cwy[f] = iyc - fy0;
    F.cgx[f] = mx ? P.sx * inv : 0.0f;
    F.cgy[f] = my ? P.sy * inv : 0.0f;
  }
}

template <class C, bool WITH_ID = true, int ROW_STEP = 1, bool TG_DIRECT = false>
MD2_HD void stage_a_issue(Lane<C>& L, const Params& P, const WarpJob& J, int t) {
  stage_a_issue<C, WITH_ID, ROW_STEP, TG_DIRECT>(L, L.fl, P, J, t);
}

// stage_a_finish: the taps have arrived; interpolate pred and its derivatives, export pr/tg for
// the neighbour exchange and stash what the adjoint of row t needs later.
// PUBLISH: the row's target / pred fields go to the ring even without gradients (the role-specialised
// kernel hands rows from warp to warp through it)
template <class C, class ST, bool PUBLISH = C::GRAD>
MD2_HD void stage_a_finish(Lane<C>& L, const Flight<C>& F, const Params& P, const WarpJob& J, int t, const ST& st) {
  const int slot = st.slot(t);
  const F4 tg4 = F.ctg;
  const float z = F.cz;
  const bool own = (t >= J.y0) && (t < J.y1) && (L.x >= J.x0) && (L.x < J.x0 + kOwnCols) && L.colok;
  L.tg[0] = tg4.x; L.tg[1] = tg4.y; L.tg[2] = tg4.z;
  if (own) MD2_CHK(t * J.W + L.xi, J.plane);
  if (J.depth && own) J.depth[t * J.W + L.xi] = z;
  // WarpJob::staged: field 0 (the target texels) is written by the TMA copy of the row and by nobody else
  if (PUBLISH && !J.staged) st.at(slot, 0, C::STASH4) = make_f4(tg4.x, tg4.y, tg4.z, 0.f);
#pragma unroll
  for (int f = 0; f < C::NSRC; ++f) {
    const F4 nw = F.tap[f][0], ne = F.tap[f][1], sw = F.tap[f][2], se = F.tap[f][3];
    const float wx = F.cwx[f], wy = F.cwy[f], gxs = F.cgx[f], gys = F.cgy[f];
    float pr[3], dxp[3], dyp[3];
    {
      const float nwc[3] = {nw.x, nw.y, nw.z}, nec[3] = {ne.x, ne.y, ne.z};
      const float swc[3] = {sw.x, sw.y, sw.z}, sec[3] = {se.x, se.y, se.z};
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float dn = nec[c] - nwc[c], ds = sec[c] - swc[c];
        const float top = fmaf(wx, dn, nwc[c]), bot = fmaf(wx, ds, swc[c]);
        const float dv = bot - top;
        pr[c] = fmaf(wy, dv, top);
        dxp[c] = fmaf(wy, ds - dn, dn) * gxs;
        dyp[c] = dv * gys;
      }
    }
    if (J.warped[f] && own) {
#pragma unroll
      for (int c = 0; c < 3; ++c) J.warped[f][c * J.plane + t * J.W + L.xi] = pr[c];
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) L.pr[f][c] = pr[c];
    if (PUBLISH) st.at(slot, 1 + 3 * f, C::STASH4) = make_f4(pr[0], pr[1], pr[2], F.cu[f]);
    if (C::GRAD) {
      st.at(slot, 2 + 3 * f, C::STASH4) = make_f4(dxp[0], dxp[1], dxp[2], F.cv[f]);
      st.at(slot, 3 + 3 * f, C::STASH4) = make_f4(dyp[0], dyp[1], dyp[2], f == 0 ? z : 0.f);   // depth rides with source 0
    }
  }
}

template <class C, class ST, bool PUBLISH = C::GRAD>
MD2_HD void stage_a_finish(Lane<C>& L, const Params& P, const WarpJob& J, int t, const ST& st) {
  stage_a_finish<C, ST, PUBLISH>(L, L.fl, P, J, t, st);
}

// ------------------------------------------------------------------ stage B
// Horizontal sums of row t, SSIM + L1 of window row t-1, per-pixel minimum and the
// SSIM-adjoint coefficients of the winning source.
template <class C>
MD2_HD void stage_b_divergent(Lane<C>& L, const Params& P, const WarpJob& J, int t, int lane,
                    const Xchg1<C>& lf, const Xchg1<C>& rt) {
  const int yw = t - 1;
  float H0[C::NSRC][3][3], HY0[3][2];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float yl = lf.tg[c], yr = rt.tg[c], yc = L.tg[c];
    HY0[c][0] = yl + yc + yr;
    HY0[c][1] = fmaf(yr, yr, fmaf(yc, yc, yl * yl));
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f) {
      const float xl = lf.pr[f][c], xr = rt.pr[f][c], xc = L.pr[f][c];
      H0[f][c][0] = xl + xc + xr;
      H0[f][c][1] = fmaf(xr, xr, fmaf(xc, xc, xl * xl));
      H0[f][c][2] = fmaf(xr, yr, fmaf(xc, yc, xl * yl));
    }
  }
  // windows this job needs: its own rows plus one halo row each side (for the adjoint)
  const bool win_ok = L.colok && (yw >= 0) && (yw < P.H) && (lane >= 1) && (lane <= kLanes - 2) &&
                      (yw >= J.y0 - (C::GRAD ? 1 : 0)) && (yw < J.y1 + (C::GRAD ? 1 : 0));
  const bool own_win = win_ok && (lane >= 2) && (lane < 2 + kOwnCols) && (yw >= J.y0) && (yw < J.y1);
  int tag = -1;
#pragma unroll
  for (int n = 0; n < C::NCS; ++n)
#pragma unroll
    for (int k = 0; k < 9; ++k) L.coef[n][k] = 0.f;
  if (win_ok) {
    float V[C::NSRC][3][3], VY[3][2];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      // H2 / HY2 hold the SUM of the two previous rows (one add here, one add and one move below)
#pragma unroll
      for (int k = 0; k < 2; ++k) VY[c][k] = L.HY2[c][k] + HY0[c][k];
#pragma unroll
      for (int f = 0; f < C::NSRC; ++f)
#pragma unroll
        for (int k = 0; k < 3; ++k) V[f][c][k] = L.H2[f][c][k] + H0[f][c][k];
    }
    float rl[C::NSRC];
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f) {
      float ss = 0.f, l1 = 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        if (!C::NOSSIM) ss += ssim_window(V[f][c][0], V[f][c][1], V[f][c][2], VY[c][0], VY[c][1], nullptr);
        l1 += fabsf(L.tg1[c] - L.pr1[f][c]);
      }
      // trainer.py:403: 0.85 * ssim.mean(1) + 0.15 * l1.mean(1)   (--no_ssim: l1.mean(1), :399-400)
      rl[f] = C::NOSSIM ? l1 * (1.0f / 3.0f) : fmaf(0.85f / 3.0f, ss, (0.15f / 3.0f) * l1);
    }
    // candidates in the order of trainer.py:471: identity first, then reprojection
    float best = INFINITY;
    if (C::AUTOMASK) {
      if (C::AVG) {
        float acc = 0.f;
#pragma unroll
        for (int f = 0; f < C::NSRC; ++f) acc += L.idv[f];
        best = MD2_FADD(acc * (1.0f / (float)C::NSRC), MD2_FMUL(L.nzv[0], 0.00001f));
      } else {
#pragma unroll
        for (int f = 0; f < C::NSRC; ++f) {
          const float cand = MD2_FADD(L.idv[f], MD2_FMUL(L.nzv[f], 0.00001f));
          if (cand < best) best = cand;
        }
      }
    }
    float rlm[C::NSRC];
    pmask_apply<C>(L, J, rl, rlm);
    if (C::AVG) {
      float acc = 0.f;
#pragma unroll
      for (int f = 0; f < C::NSRC; ++f) acc += rlm[f];
      const float cand = acc * (1.0f / (float)C::NSRC);
      if (cand < best) { best = cand; tag = 0; }
    } else {
#pragma unroll
      for (int f = 0; f < C::NSRC; ++f)
        if (rlm[f] < best) { best = rlm[f]; tag = f; }
    }
    if (own_win) {
      L.loss += best;
      MD2_CHK(yw * J.W + L.xi, J.plane);
      if (C::AUTOMASK && J.idsel) J.idsel[yw * J.W + L.xi] = (tag >= 0) ? 1.0f : 0.0f;
    }
    if (C::GRAD && !C::NOSSIM && tag >= 0) {
      if (C::AVG) {
#pragma unroll
        for (int f = 0; f < C::NSRC; ++f)
#pragma unroll
          for (int c = 0; c < 3; ++c)
          {
            unsigned char* lp = nullptr;
            MD2_DBG(lp = (L.colok && yw >= 0 && yw < J.H)
                        ? &D.live[(((((long)J.s * D.B + J.b) * D.nsrc + f) * 3 + c) * D.H + yw) * D.W + L.x] : nullptr;);
            ssim_window(V[f][c][0], V[f][c][1], V[f][c][2], VY[c][0], VY[c][1], &L.coef[f][c * 3], true, lp);
          }
      } else {
        // select the winner's window sums without dynamic register indexing
        float W3[3][3];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            float v = V[0][c][k];
#pragma unroll
            for (int f = 1; f < C::NSRC; ++f) v = (tag == f) ? V[f][c][k] : v;
            W3[c][k] = v;
          }
#pragma unroll
        for (int c = 0; c < 3; ++c)
        {
          unsigned char* lp = nullptr;
          MD2_DBG(lp = (tag >= 0 && L.colok && yw >= 0 && yw < J.H)
                      ? &D.live[(((((long)J.s * D.B + J.b) * D.nsrc + tag) * 3 + c) * D.H + yw) * D.W + L.x] : nullptr;);
          ssim_window(W3[c][0], W3[c][1], W3[c][2], VY[c][0], VY[c][1], &L.coef[0][c * 3], true, lp);
        }
      }
    }
    pmask_backward<C>(L, P, J, rl, tag, own_win, yw);
  }
  L.tag = tag;
  MD2_DBG(if (own_win) D.tag[(((long)J.s * D.B + J.b) * D.H + yw) * D.W + L.x] = (signed char)tag;);
  // roll the forward state
#pragma unroll
  for (int c = 0; c < 3; ++c) {
#pragma unroll
    for (int k = 0; k < 2; ++k) { L.HY2[c][k] = L.HY1[c][k] + HY0[c][k]; L.HY1[c][k] = HY0[c][k]; }
    L.tg1[c] = L.tg[c];
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f) {
#pragma unroll
      for (int k = 0; k < 3; ++k) { L.H2[f][c][k] = L.H1[f][c][k] + H0[f][c][k]; L.H1[f][c][k] = H0[f][c][k]; }
      L.pr1[f][c] = L.pr[f][c];
    }
  }
}

template <class C>
MD2_HD void stage_b_straight(Lane<C>& L, const Params& P, const WarpJob& J, int t, int lane,
                    const Xchg1<C>& lf, const Xchg1<C>& rt) {
  const int yw = t - 1;
  float H0[C::NSRC][3][3], HY0[3][2];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float yl = lf.tg[c], yr = rt.tg[c], yc = L.tg[c];
    HY0[c][0] = yl + yc + yr;
    HY0[c][1] = fmaf(yr, yr, fmaf(yc, yc, yl * yl));
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f) {
      const float xl = lf.pr[f][c], xr = rt.pr[f][c], xc = L.pr[f][c];
      H0[f][c][0] = xl + xc + xr;
      H0[f][c][1] = fmaf(xr, xr, fmaf(xc, xc, xl * xl));
      H0[f][c][2] = fmaf(xr, yr, fmaf(xc, yc, xl * yl));
    }
  }
  // windows this job needs: its own rows plus one halo row each side (for the adjoint)
  const bool win_ok = L.colok && (yw >= 0) && (yw < P.H) && (lane >= 1) && (lane <= kLanes - 2) &&
                      (yw >= J.y0 - (C::GRAD ? 1 : 0)) && (yw < J.y1 + (C::GRAD ? 1 : 0));
  const bool own_win = win_ok && (lane >= 2) && (lane < 2 + kOwnCols) && (yw >= J.y0) && (yw < J.y1);
  // Cfg::STRAIGHT: lanes / rows that do not need the window compute it anyway (the warp executes the
  // code as long as one lane needs it) and are masked at the end, which avoids a divergent region and
  // the register copies at its join; otherwise the block is skipped by the lanes that do not need it.
  int tag = -1;
  {
    float V[C::NSRC][3][3], VY[3][2];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      // H2 / HY2 hold the SUM of the two previous rows (one add here, one add and one move below)
#pragma unroll
      for (int k = 0; k < 2; ++k) VY[c][k] = L.HY2[c][k] + HY0[c][k];
#pragma unroll
      for (int f = 0; f < C::NSRC; ++f)
#pragma unroll
        for (int k = 0; k < 3; ++k) V[f][c][k] = L.H2[f][c][k] + H0[f][c][k];
    }
    float rl[C::NSRC];
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f) {
      float ss = 0.f, l1 = 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        if (!C::NOSSIM) ss += ssim_window(V[f][c][0], V[f][c][1], V[f][c][2], VY[c][0], VY[c][1], nullptr);
        l1 += fabsf(L.tg1[c] - L.pr1[f][c]);
      }
      // trainer.py:403: 0.85 * ssim.mean(1) + 0.15 * l1.mean(1)   (--no_ssim: l1.mean(1), :399-400)
      rl[f] = C::NOSSIM ? l1 * (1.0f / 3.0f) : fmaf(0.85f / 3.0f, ss, (0.15f / 3.0f) * l1);
    }
    // candidates in the order of trainer.py:471: identity first, then reprojection
    float best = INFINITY;
    if (C::AUTOMASK) {
      if (C::AVG) {
        float acc = 0.f;
#pragma unroll
        for (int f = 0; f < C::NSRC; ++f) acc += L.idv[f];
        best = MD2_FADD(acc * (1.0f / (float)C::NSRC), MD2_FMUL(L.nzv[0], 0.00001f));
      } else {
#pragma unroll
        for (int f = 0; f < C::NSRC; ++f) {
          const float cand = MD2_FADD(L.idv[f], MD2_FMUL(L.nzv[f], 0.00001f));
          best = (cand < best) ? cand : best;
        }
      }
    }
    float rlm[C::NSRC];
    pmask_apply<C>(L, J, rl, rlm);
    if (C::AVG) {
      float acc = 0.f;
#pragma unroll
      for (int f = 0; f < C::NSRC; ++f) acc += rlm[f];
      const float cand = acc * (1.0f / (float)C::NSRC);
      tag = (cand < best) ? 0 : tag;
      best = (cand < best) ? cand : best;
    } else {
#pragma unroll
      for (int f = 0; f < C::NSRC; ++f) {
        tag = (rlm[f] < best) ? f : tag;
        best = (rlm[f] < best) ? rlm[f] : best;
      }
    }
    tag = win_ok ? tag : -1;
    L.loss += own_win ? best : 0.0f;
    if (own_win) MD2_CHK(yw * J.W + L.xi, J.plane);
    if (C::AUTOMASK && J.idsel && own_win) J.idsel[yw * J.W + L.xi] = (tag >= 0) ? 1.0f : 0.0f;
    if (C::GRAD && !C::NOSSIM) {
      const bool valid = tag >= 0;
      if (C::AVG) {
#pragma unroll
        for (int f = 0; f < C::NSRC; ++f)
#pragma unroll
          for (int c = 0; c < 3; ++c)
          {
            unsigned char* lp = nullptr;
            MD2_DBG(lp = (valid && L.colok && yw >= 0 && yw < J.H)
                        ? &D.live[(((((long)J.s * D.B + J.b) * D.nsrc + f) * 3 + c) * D.H + yw) * D.W + L.x] : nullptr;);
            ssim_window(V[f][c][0], V[f][c][1], V[f][c][2], VY[c][0], VY[c][1], &L.coef[f][c * 3], valid, lp);
          }
      } else {
        // select the winner's window sums without dynamic register indexing
        float W3[3][3];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            float v = V[0][c][k];
#pragma unroll
            for (int f = 1; f < C::NSRC; ++f) v = (tag == f) ? V[f][c][k] : v;
            W3[c][k] = v;
          }
#pragma unroll
        for (int c = 0; c < 3; ++c)
        {
          unsigned char* lp = nullptr;
          MD2_DBG(lp = (tag >= 0 && L.colok && yw >= 0 && yw < J.H)
                      ? &D.live[(((((long)J.s * D.B + J.b) * D.nsrc + tag) * 3 + c) * D.H + yw) * D.W + L.x] : nullptr;);
          ssim_window(W3[c][0], W3[c][1], W3[c][2], VY[c][0], VY[c][1], &L.coef[0][c * 3], valid, lp);
        }
      }
    } else {
#pragma unroll
      for (int n = 0; n < C::NCS; ++n)
#pragma unroll
        for (int k = 0; k < 9; ++k) L.coef[n][k] = 0.f;
    }
    pmask_backward<C>(L, P, J, rl, tag, own_win, yw);
  }
  L.tag = tag;
  MD2_DBG(if (own_win) D.tag[(((long)J.s * D.B + J.b) * D.H + yw) * D.W + L.x] = (signed char)tag;);
  // roll the forward state
#pragma unroll
  for (int c = 0; c < 3; ++c) {
#pragma unroll
    for (int k = 0; k < 2; ++k) { L.HY2[c][k] = L.HY1[c][k] + HY0[c][k]; L.HY1[c][k] = HY0[c][k]; }
    L.tg1[c] = L.tg[c];
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f) {
#pragma unroll
      for (int k = 0; k < 3; ++k) { L.H2[f][c][k] = L.H1[f][c][k] + H0[f][c][k]; L.H1[f][c][k] = H0[f][c][k]; }
      L.pr1[f][c] = L.pr[f][c];
    }
  }
}

// Two control-flow shapes of the same arithmetic (Cfg::STRAIGHT): "divergent" skips the window /
// pixel block for the lanes that do not need it, "straight" lets every lane compute and masks the
// results (no divergent region, no register copies at its join).  Measured on B200 (r01 log): with 3
// sources straight is 7 % faster, with 1-2 sources divergent is 3 % faster.
template <class C>
MD2_HD void stage_b(Lane<C>& L, const Params& P, const WarpJob& J, int t, int lane,
                    const Xchg1<C>& lf, const Xchg1<C>& rt) {
  if (C::STRAIGHT) stage_b_straight(L, P, J, t, lane, lf, rt);
  else stage_b_divergent(L, P, J, t, lane, lf, rt);
}

// ------------------------------------------------------------------ stage C
// Adjoint for pixel row t-2: 3x3 box adjoint of the coefficient maps (with the fold
// of the reflection ring, SURVEY.md A.2), d loss/d pred, grid-sample and projection
// adjoints (A.3).  Writes d loss / d D for owned pixels and accumulates the pose sums.
template <class C, class ST>
MD2_HD void stage_c_divergent(Lane<C>& L, const Params& P, const WarpJob& J, int t, int lane,
                    const Xchg2<C>& lf, const Xchg2<C>& rt, const ST& st) {
  const int yp = t - 2;
  const float wl = (L.x == 1) ? 2.0f : 1.0f;
  const float wr = (L.x == P.W - 2) ? 2.0f : 1.0f;
  float B0[C::NSRC][9];
#pragma unroll
  for (int f = 0; f < C::NSRC; ++f) {
    const int n = C::AVG ? f : 0;
    const float ml = (C::AVG || lf.tag == f) ? wl : 0.0f;
    const float mc = (C::AVG || L.tag == f) ? 1.0f : 0.0f;
    const float mr = (C::AVG || rt.tag == f) ? wr : 0.0f;
#pragma unroll
    for (int k = 0; k < 9; ++k)
      B0[f][k] = fmaf(ml, lf.coef[n][k], fmaf(mr, rt.coef[n][k], mc * L.coef[n][k]));
  }
  const bool own = L.colok && (lane >= 2) && (lane < 2 + kOwnCols) && (yp >= J.y0) && (yp < J.y1);
  const int bslot = t & 1;          // ring slot of row t (holds row t-2 until overwritten below)
  if (own) {
    float B1v[C::NSRC][9], B2v[C::NSRC][9];
    if (C::BSMEM) {
      float f1[4 * C::NB4], f2[4 * C::NB4];
#pragma unroll
      for (int i = 0; i < C::NB4; ++i) {
        const F4 a = st.b(bslot ^ 1, i, C::NB4), c2 = st.b(bslot, i, C::NB4);
        f1[4 * i] = a.x; f1[4 * i + 1] = a.y; f1[4 * i + 2] = a.z; f1[4 * i + 3] = a.w;
        f2[4 * i] = c2.x; f2[4 * i + 1] = c2.y; f2[4 * i + 2] = c2.z; f2[4 * i + 3] = c2.w;
      }
#pragma unroll
      for (int f = 0; f < C::NSRC; ++f)
#pragma unroll
        for (int k = 0; k < 9; ++k) { B1v[f][k] = f1[f * 9 + k]; B2v[f][k] = f2[f * 9 + k]; }
    } else {
#pragma unroll
      for (int f = 0; f < C::NSRC; ++f)
#pragma unroll
        for (int k = 0; k < 9; ++k) { B1v[f][k] = L.B1[f][k]; B2v[f][k] = L.B2[f][k]; }
    }
    const float wu = (yp == 1) ? 2.0f : 1.0f;
    const float wd = (yp == P.H - 2) ? 2.0f : 1.0f;
    const int slot = st.slot(yp);
    const F4 s0 = st.at(slot, 0, C::STASH4);
    const float tg[3] = {s0.x, s0.y, s0.z};
    const float z = st.at(slot, 3, C::STASH4).w;
    const float yf = (float)yp;
    float dzsum = 0.f;
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f) {
      F4 sp = st.at(slot, 1 + 3 * f, C::STASH4);
      if (C::PAIRED) {
        const F4 a = st.at(slot, 1, C::STASH4), b4 = st.at(slot, 4, C::STASH4);
        sp = f == 0 ? make_f4(a.x, a.y, b4.x, b4.z) : make_f4(a.z, a.w, b4.y, b4.w);
      }
      const F4 sdx = st.at(slot, 2 + 3 * f, C::STASH4);
      const F4 sdy = st.at(slot, 3 + 3 * f, C::STASH4);
      const float xs[3] = {sp.x, sp.y, sp.z};
      const float dxs[3] = {sdx.x, sdx.y, sdx.z}, dys[3] = {sdy.x, sdy.y, sdy.z};
      const bool won = C::AVG ? (L.tag1 >= 0) : (L.tag1 == f);
      // --predictive_mask: the L1 term of this pixel carries its mask value (the SSIM coefficients already do)
      const float mk = (!C::AUTOMASK && J.pm && won) ? MD2_LD(J.pm + f * J.plane + yp * J.W + L.xi) : 1.0f;
      float d0 = 0.f, d1 = 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float xj = xs[c];
        const float A = fmaf(wu, B2v[f][c * 3 + 0], fmaf(wd, B0[f][c * 3 + 0], B1v[f][c * 3 + 0]));
        const float Bq = fmaf(wu, B2v[f][c * 3 + 1], fmaf(wd, B0[f][c * 3 + 1], B1v[f][c * 3 + 1]));
        const float G = fmaf(wu, B2v[f][c * 3 + 2], fmaf(wd, B0[f][c * 3 + 2], B1v[f][c * 3 + 2]));
        // d loss / d pred_c = 0.85/3 * SSIM part + 0.15/3 * sign(x - y) [if this source won here]
        float g = C::NOSSIM ? 0.0f : (0.85f / 3.0f) * fmaf(xj, Bq, fmaf(tg[c], G, A));
        if (won) {
          const float kl1 = (C::NOSSIM ? (1.0f / 3.0f) : (0.15f / 3.0f)) * mk;
          const float df = xj - tg[c];
          g += (df != 0.f) ? copysignf(kl1, df) : 0.0f;
          MD2_DBG(D.l1sgn[(((((long)J.s * D.B + J.b) * D.nsrc + f) * 3 + c) * D.H + yp) * D.W + L.x] =
                      (signed char)(df > 0.f ? 1 : (df < 0.f ? -1 : 0)););
        }
        d0 = fmaf(g, dxs[c], d0);
        d1 = fmaf(g, dys[c], d1);
      }
      const float u = sp.w, v = sdx.w;
      const float d2 = -fmaf(u, d0, v * d1);
      const float q0 = fmaf(L.qb[f][0], yf, L.qa[f][0]);
      const float q1 = fmaf(L.qb[f][1], yf, L.qa[f][1]);
      const float q2 = fmaf(L.qb[f][2], yf, L.qa[f][2]);
      dzsum += fmaf(d0, q0, fmaf(d1, q1, d2 * q2));
      const float zy = z * yf;
      L.S1[f][0] = fmaf(d0, z, L.S1[f][0]); L.S1[f][1] = fmaf(d1, z, L.S1[f][1]); L.S1[f][2] = fmaf(d2, z, L.S1[f][2]);
      L.S2[f][0] = fmaf(d0, zy, L.S2[f][0]); L.S2[f][1] = fmaf(d1, zy, L.S2[f][1]); L.S2[f][2] = fmaf(d2, zy, L.S2[f][2]);
      L.S3[f][0] += d0; L.S3[f][1] += d1; L.S3[f][2] += d2;
    }
    // d depth / d D = -c * z^2  (layers.py:23-24)
    const float dD = -P.c_disp * z * z * dzsum * P.gscale;
    MD2_CHK(yp * J.W + L.xi, J.plane);
    J.dD[yp * J.W + L.xi] = dD;
    if (J.s == 0)   // up-sampling is the identity at scale 0: finish grad_disp_0 here (A.4 + A.3)
      J.gd0[yp * J.W + L.xi] = dD + J.sm_w * (MD2_LD(J.gn0 + yp * J.W + L.xi) * J.sm_inv_m - J.sm_dterm);
  }
  if (C::BSMEM) {
    float fl[4 * C::NB4];
#pragma unroll
    for (int i = 0; i < 4 * C::NB4; ++i) fl[i] = 0.f;
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f)
#pragma unroll
      for (int k = 0; k < 9; ++k) fl[f * 9 + k] = B0[f][k];
#pragma unroll
    for (int i = 0; i < C::NB4; ++i)
      st.b(bslot, i, C::NB4) = make_f4(fl[4 * i], fl[4 * i + 1], fl[4 * i + 2], fl[4 * i + 3]);
  } else {
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f)
#pragma unroll
      for (int k = 0; k < 9; ++k) { L.B2[f][k] = L.B1[f][k]; L.B1[f][k] = B0[f][k]; }
  }
  L.tag1 = L.tag;
}

template <class C, class ST>
MD2_HD void stage_c_straight(Lane<C>& L, const Params& P, const WarpJob& J, int t, int lane,
                    const Xchg2<C>& lf, const Xchg2<C>& rt, const ST& st) {
  const int yp = t - 2;
  const float wl = (L.x == 1) ? 2.0f : 1.0f;
  const float wr = (L.x == P.W - 2) ? 2.0f : 1.0f;
  float B0[C::NSRC][9];
#pragma unroll
  for (int f = 0; f < C::NSRC; ++f) {
    const int n = C::AVG ? f : 0;
    const float ml = (C::AVG || lf.tag == f) ? wl : 0.0f;
    const float mc = (C::AVG || L.tag == f) ? 1.0f : 0.0f;
    const float mr = (C::AVG || rt.tag == f) ? wr : 0.0f;
#pragma unroll
    for (int k = 0; k < 9; ++k)
      B0[f][k] = fmaf(ml, lf.coef[n][k], fmaf(mr, rt.coef[n][k], mc * L.coef[n][k]));
  }
  const bool own = L.colok && (lane >= 2) && (lane < 2 + kOwnCols) && (yp >= J.y0) && (yp < J.y1);
  const int bslot = t & 1;          // ring slot of row t (holds row t-2 until overwritten below)
  // Cfg::STRAIGHT (see stage_b): every lane computes, only owners accumulate and store
  {
    float B1v[C::NSRC][9], B2v[C::NSRC][9];
    if (C::BSMEM) {
      float f1[4 * C::NB4], f2[4 * C::NB4];
#pragma unroll
      for (int i = 0; i < C::NB4; ++i) {
        const F4 a = st.b(bslot ^ 1, i, C::NB4), c2 = st.b(bslot, i, C::NB4);
        f1[4 * i] = a.x; f1[4 * i + 1] = a.y; f1[4 * i + 2] = a.z; f1[4 * i + 3] = a.w;
        f2[4 * i] = c2.x; f2[4 * i + 1] = c2.y; f2[4 * i + 2] = c2.z; f2[4 * i + 3] = c2.w;
      }
#pragma unroll
      for (int f = 0; f < C::NSRC; ++f)
#pragma unroll
        for (int k = 0; k < 9; ++k) { B1v[f][k] = f1[f * 9 + k]; B2v[f][k] = f2[f * 9 + k]; }
    } else {
#pragma unroll
      for (int f = 0; f < C::NSRC; ++f)
#pragma unroll
        for (int k = 0; k < 9; ++k) { B1v[f][k] = L.B1[f][k]; B2v[f][k] = L.B2[f][k]; }
    }
    const float wu = (yp == 1) ? 2.0f : 1.0f;
    const float wd = (yp == P.H - 2) ? 2.0f : 1.0f;
    const int slot = st.slot(yp);
    const F4 s0 = st.at(slot, 0, C::STASH4);
    const float tg[3] = {s0.x, s0.y, s0.z};
    // (select: rows t0 - 2, t0 - 1 of the ring are never written, and 0 * stale non-finite z would poison the pose sums)
    const float z = own ? st.at(slot, 3, C::STASH4).w : 0.0f;
    const float yf = (float)yp;
    float dzsum = 0.f;
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f) {
      F4 sp = st.at(slot, 1 + 3 * f, C::STASH4);
      if (C::PAIRED) {
        const F4 a = st.at(slot, 1, C::STASH4), b4 = st.at(slot, 4, C::STASH4);
        sp = f == 0 ? make_f4(a.x, a.y, b4.x, b4.z) : make_f4(a.z, a.w, b4.y, b4.w);
      }
      const F4 sdx = st.at(slot, 2 + 3 * f, C::STASH4);
      const F4 sdy = st.at(slot, 3 + 3 * f, C::STASH4);
      const float xs[3] = {sp.x, sp.y, sp.z};
      const float dxs[3] = {sdx.x, sdx.y, sdx.z}, dys[3] = {sdy.x, sdy.y, sdy.z};
      const bool won = C::AVG ? (L.tag1 >= 0) : (L.tag1 == f);
      const float mk = (!C::AUTOMASK && J.pm && won && own) ? MD2_LD(J.pm + f * J.plane + yp * J.W + L.xi) : 1.0f;
      float d0 = 0.f, d1 = 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float xj = xs[c];
        const float A = fmaf(wu, B2v[f][c * 3 + 0], fmaf(wd, B0[f][c * 3 + 0], B1v[f][c * 3 + 0]));
        const float Bq = fmaf(wu, B2v[f][c * 3 + 1], fmaf(wd, B0[f][c * 3 + 1], B1v[f][c * 3 + 1]));
        const float G = fmaf(wu, B2v[f][c * 3 + 2], fmaf(wd, B0[f][c * 3 + 2], B1v[f][c * 3 + 2]));
        // d loss / d pred_c = 0.85/3 * SSIM part + 0.15/3 * sign(x - y) [if this source won here]
        float g = C::NOSSIM ? 0.0f : (0.85f / 3.0f) * fmaf(xj, Bq, fmaf(tg[c], G, A));
        {
          const float kl1 = (C::NOSSIM ? (1.0f / 3.0f) : (0.15f / 3.0f)) * mk;
          const float df = xj - tg[c];
          g += (won && df != 0.f) ? copysignf(kl1, df) : 0.0f;
          MD2_DBG(if (own) D.l1sgn[(((((long)J.s * D.B + J.b) * D.nsrc + f) * 3 + c) * D.H + yp) * D.W + L.x] =
                      (signed char)(df > 0.f ? 1 : (df < 0.f ? -1 : 0)););
        }
        d0 = fmaf(g, dxs[c], d0);
        d1 = fmaf(g, dys[c], d1);
      }
      d0 = own ? d0 : 0.0f;      // selects, not products: non-owners may hold stale (non-finite) stash
      d1 = own ? d1 : 0.0f;
      const float u = sp.w, v = sdx.w;
      const float d2 = own ? -fmaf(u, d0, v * d1) : 0.0f;
      const float q0 = fmaf(L.qb[f][0], yf, L.qa[f][0]);
      const float q1 = fmaf(L.qb[f][1], yf, L.qa[f][1]);
      const float q2 = fmaf(L.qb[f][2], yf, L.qa[f][2]);
      dzsum += fmaf(d0, q0, fmaf(d1, q1, d2 * q2));
      const float zy = z * yf;
      L.S1[f][0] = fmaf(d0, z, L.S1[f][0]); L.S1[f][1] = fmaf(d1, z, L.S1[f][1]); L.S1[f][2] = fmaf(d2, z, L.S1[f][2]);
      L.S2[f][0] = fmaf(d0, zy, L.S2[f][0]); L.S2[f][1] = fmaf(d1, zy, L.S2[f][1]); L.S2[f][2] = fmaf(d2, zy, L.S2[f][2]);
      L.S3[f][0] += d0; L.S3[f][1] += d1; L.S3[f][2] += d2;
    }
    // d depth / d D = -c * z^2  (layers.py:23-24)
    const float dD = -P.c_disp * z * z * dzsum * P.gscale;
    if (own) {
      MD2_CHK(yp * J.W + L.xi, J.plane);
      J.dD[yp * J.W + L.xi] = dD;
      if (J.s == 0)   // up-sampling is the identity at scale 0: finish grad_disp_0 here (A.4 + A.3)
        J.gd0[yp * J.W + L.xi] = dD + J.sm_w * (MD2_LD(J.gn0 + yp * J.W + L.xi) * J.sm_inv_m - J.sm_dterm);
    }
  }
  if (C::BSMEM) {
    float fl[4 * C::NB4];
#pragma unroll
    for (int i = 0; i < 4 * C::NB4; ++i) fl[i] = 0.f;
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f)
#pragma unroll
      for (int k = 0; k < 9; ++k) fl[f * 9 + k] = B0[f][k];
#pragma unroll
    for (int i = 0; i < C::NB4; ++i)
      st.b(bslot, i, C::NB4) = make_f4(fl[4 * i], fl[4 * i + 1], fl[4 * i + 2], fl[4 * i + 3]);
  } else {
#pragma unroll
    for (int f = 0; f < C::NSRC; ++f)
#pragma unroll
      for (int k = 0; k < 9; ++k) { L.B2[f][k] = L.B1[f][k]; L.B1[f][k] = B0[f][k]; }
  }
  L.tag1 = L.tag;
}

template <class C, class ST>
MD2_HD void stage_c(Lane<C>& L, const Params& P, const WarpJob& J, int t, int lane,
                    const Xchg2<C>& lf, const Xchg2<C>& rt, const ST& st) {
  if (C::STRAIGHT) stage_c_straight(L, P, J, t, lane, lf, rt, st);
  else stage_c_divergent(L, P, J, t, lane, lf, rt, st);
}

// Turns the lane's pose sums into its share of dP (3x4, row-major) for source f:
// dP[i][k<3] = a_k S1_i + b_k S2_i with inv_K3 (x,y,1)_k = a_k + b_k y ; dP[i][3] = S3_i.
template <class C>
MD2_HD void lane_dP(const Lane<C>& L, const Params& P, const WarpJob& J, int f, float* dP) {
  const float* ik = P.invK + (size_t)J.b * 16;
  const float xf = (float)L.xi;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float ak = fmaf(MD2_LD(ik + k * 4 + 0), xf, MD2_LD(ik + k * 4 + 2));
    const float bk = MD2_LD(ik + k * 4 + 1);
#pragma unroll
    for (int i = 0; i < 3; ++i) dP[i * 4 + k] = fmaf(ak, L.S1[f][i], bk * L.S2[f][i]);
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) dP[i * 4 + 3] = L.S3[f][i];
}

// ------------------------------------------------------------------ identity pass
// Scale-independent identity reprojection losses (trainer.py:432-439): SSIM+L1 between
// the unwarped source f and the target.  One lane per column, halo 1; rows and columns are
// read at their reflected positions.
template <int NSRC>
struct IdLane {
  int x, xi;
  bool colok;
  float H1[NSRC][3][3], H2[NSRC][3][3];
  float HY1[3][2], HY2[3][2];
  float pr1[NSRC][3], tg1[3];
  float pr[NSRC][3], tg[3];
  float npr[NSRC][3], ntg[3];     // next row, in flight
};
template <int NSRC>
struct IdXchg {
  float pr[NSRC][3];
  float tg[3];
};

template <int NSRC>
MD2_HD void id_init(IdLane<NSRC>& L, const Params& P, int x0, int lane) {
  L.x = x0 - 1 + lane;
  L.colok = (L.x >= 0) && (L.x < P.W);
  L.xi = reflect_clamp(L.x, P.W);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    L.HY1[c][0] = L.HY1[c][1] = L.HY2[c][0] = L.HY2[c][1] = 0.f;
    L.tg1[c] = L.tg[c] = 0.f;
#pragma unroll
    for (int f = 0; f < NSRC; ++f) {
      L.pr1[f][c] = L.pr[f][c] = 0.f;
#pragma unroll
      for (int k = 0; k < 3; ++k) L.H1[f][c][k] = L.H2[f][c][k] = 0.f;
    }
  }
}

// issue the planar loads of row t (target + sources, at the reflected position)
template <int NSRC>
MD2_HD void id_prefetch(IdLane<NSRC>& L, const Params& P, int b, int t) {
  const int tr = reflect_clamp(t, P.H);
  const int plane = P.H * P.W;
  const int pix = tr * P.W + L.xi;
#pragma unroll
  for (int c = 0; c < 3; ++c) L.ntg[c] = load_px(P.tgt, P.tgt8, P.u8_hwc, b, c, plane, pix);
#pragma unroll
  for (int f = 0; f < NSRC; ++f)
#pragma unroll
    for (int c = 0; c < 3; ++c) L.npr[f][c] = load_px(P.src[f], P.src8[f], P.u8_hwc, b, c, plane, pix);
}

// Consumes row t of the planar NCHW target / sources (prefetched one step earlier), puts row t+1 in
// flight and, for the pixels this lane owns, writes the RGBx texels the marching kernel gathers
// from: the re-layout costs no extra pass over the images.
template <int NSRC>
MD2_HD void id_stage_a(IdLane<NSRC>& L, const Params& P, int b, int t, int lane, int y0, int y1) {
  const int tr = reflect_clamp(t, P.H);
  const int plane = P.H * P.W;
  const bool own = L.colok && t >= y0 && t < y1 && lane >= 1 && lane <= kIdCols;
  const int o4 = 4 * (b * plane + tr * P.W + L.xi);
#pragma unroll
  for (int c = 0; c < 3; ++c) L.tg[c] = L.ntg[c];
#pragma unroll
  for (int f = 0; f < NSRC; ++f)
#pragma unroll
    for (int c = 0; c < 3; ++c) L.pr[f][c] = L.npr[f][c];
  id_prefetch(L, P, b, t + 1);
  if (own) {
    *reinterpret_cast<F4*>(P.tgt4 + o4) = make_f4(L.tg[0], L.tg[1], L.tg[2], 0.f);
#pragma unroll
    for (int f = 0; f < NSRC; ++f)
      *reinterpret_cast<F4*>(P.src4[f] + o4) = make_f4(L.pr[f][0], L.pr[f][1], L.pr[f][2], 0.f);
  }
}

template <int NSRC, bool NOSSIM = false>
MD2_HD void id_stage_b(IdLane<NSRC>& L, const Params& P, int b, int t, int lane, int y0, int y1,
                       const IdXchg<NSRC>& lf, const IdXchg<NSRC>& rt, int lane_lo = 1, int lane_hi = kIdCols) {
  const int yw = t - 1;
  float H0[NSRC][3][3], HY0[3][2];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float yl = lf.tg[c], yr = rt.tg[c], yc = L.tg[c];
    HY0[c][0] = yl + yc + yr;
    HY0[c][1] = fmaf(yr, yr, fmaf(yc, yc, yl * yl));
#pragma unroll
    for (int f = 0; f < NSRC; ++f) {
      const float xl = lf.pr[f][c], xr = rt.pr[f][c], xc = L.pr[f][c];
      H0[f][c][0] = xl + xc + xr;
      H0[f][c][1] = fmaf(xr, xr, fmaf(xc, xc, xl * xl));
      H0[f][c][2] = fmaf(xr, yr, fmaf(xc, yc, xl * yl));
    }
  }
  const bool own = L.colok && yw >= y0 && yw < y1 && lane >= lane_lo && lane <= lane_hi;
  if (own) {
    const size_t plane = (size_t)P.H * P.W;
#pragma unroll
    for (int f = 0; f < NSRC; ++f) {
      float ss = 0.f, l1 = 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float vy0 = L.HY2[c][0] + HY0[c][0];      // H2 / HY2 = sum of the two previous rows
        const float vy1 = L.HY2[c][1] + HY0[c][1];
        float vx[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) vx[k] = L.H2[f][c][k] + H0[f][c][k];
        if (!NOSSIM) ss += ssim_window(vx[0], vx[1], vx[2], vy0, vy1, nullptr);
        l1 += fabsf(L.tg1[c] - L.pr1[f][c]);
      }
      P.idloss[((size_t)b * NSRC + f) * plane + (size_t)yw * P.W + L.xi] =
          NOSSIM ? l1 * (1.0f / 3.0f) : fmaf(0.85f / 3.0f, ss, (0.15f / 3.0f) * l1);
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
#pragma unroll
    for (int k = 0; k < 2; ++k) { L.HY2[c][k] = L.HY1[c][k] + HY0[c][k]; L.HY1[c][k] = HY0[c][k]; }
    L.tg1[c] = L.tg[c];
#pragma unroll
    for (int f = 0; f < NSRC; ++f) {
#pragma unroll
      for (int k = 0; k < 3; ++k) { L.H2[f][c][k] = L.H1[f][c][k] + H0[f][c][k]; L.H1[f][c][k] = H0[f][c][k]; }
      L.pr1[f][c] = L.pr[f][c];
    }
  }
}

// Re-layout of one pixel of image `img` (0 = target, 1+f = source f) from planar NCHW to RGBx.
MD2_HD void pack_pixel(const Params& P, int img, int b, int p) {
  const int plane = P.H * P.W;
  const float* in = (img == 0 ? P.tgt : P.src[img - 1]);
  const unsigned char* in8 = (img == 0 ? P.tgt8 : P.src8[img - 1]);
  float* out = (img == 0 ? P.tgt4 : P.src4[img - 1]) + ((size_t)b * plane + p) * 4;
  *reinterpret_cast<F4*>(out) = make_f4(load_px(in, in8, P.u8_hwc, b, 0, plane, p), load_px(in, in8, P.u8_hwc, b, 1, plane, p),
                                        load_px(in, in8, P.u8_hwc, b, 2, plane, p), 0.f);
}

// ------------------------------------------------------------------ pose parameterisation
// transformation_from_parameters (layers.py:28-45) = rot_from_axisangle (layers.py:64-103) and
// get_translation_matrix (layers.py:48-61): T = Trans(t) R, or R^T Trans(-t) when `invert` (frame_id < 0,
// trainer.py:294-295), in fp32 like the reference; and its adjoint (where the pose gradient leaves the path).
struct Rod { float x, y, z, ca, sa, C, angle, a; };
MD2_HD Rod rodrigues(const float* v, float R[3][3]) {
  Rod r;
  r.angle = sqrtf(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
  r.a = r.angle + 1e-7f;
  r.x = v[0] / r.a; r.y = v[1] / r.a; r.z = v[2] / r.a;
  r.ca = cosf(r.angle); r.sa = sinf(r.angle); r.C = 1.f - r.ca;
  const float x = r.x, y = r.y, z = r.z, ca = r.ca, sa = r.sa, C = r.C;
  R[0][0] = x * x * C + ca; R[0][1] = x * y * C - z * sa; R[0][2] = z * x * C + y * sa;
  R[1][0] = x * y * C + z * sa; R[1][1] = y * y * C + ca; R[1][2] = y * z * C - x * sa;
  R[2][0] = z * x * C - y * sa; R[2][1] = y * z * C + x * sa; R[2][2] = z * z * C + ca;
  return r;
}
// v, t: 3 floats each; o: 16 floats (row-major 4x4)
MD2_HD void pose_to_matrix(const float* v, const float* t, int invert, float* o) {
  float R[3][3];
  rodrigues(v, R);
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) o[i * 4 + j] = invert ? R[j][i] : R[i][j];
    // invert: R^T Trans(-t) -> last column = -R^T t ; else Trans(t) R -> last column = t
    o[i * 4 + 3] = invert ? -(R[0][i] * t[0] + R[1][i] * t[1] + R[2][i] * t[2]) : t[i];
  }
  o[12] = 0.f; o[13] = 0.f; o[14] = 0.f; o[15] = 1.f;
}
// g: d loss / d T (16 floats) -> gaa, gtr (3 floats each)
MD2_HD void pose_to_matrix_backward(const float* g, const float* v, const float* t, int invert, float* gaa, float* gtr) {
  float R[3][3];
  const Rod r = rodrigues(v, R);
  float gR[3][3], gt[3];
  for (int i = 0; i < 3; ++i) {
    gt[i] = 0.f;
    for (int j = 0; j < 3; ++j) gR[i][j] = invert ? g[j * 4 + i] : g[i * 4 + j];
  }
  if (invert) {
    // col_i = -sum_k R[k][i] t[k]
    for (int i = 0; i < 3; ++i)
      for (int k = 0; k < 3; ++k) { gR[k][i] -= g[i * 4 + 3] * t[k]; gt[k] -= g[i * 4 + 3] * R[k][i]; }
  } else {
    for (int i = 0; i < 3; ++i) gt[i] = g[i * 4 + 3];
  }
  const float x = r.x, y = r.y, z = r.z, sa = r.sa, C = r.C;
  float gx = 0, gy = 0, gz = 0, gca = 0, gsa = 0, gC = 0;
  // R00 = x x C + ca
  gx += gR[0][0] * 2 * x * C; gC += gR[0][0] * x * x; gca += gR[0][0];
  // R01 = x y C - z sa
  gx += gR[0][1] * y * C; gy += gR[0][1] * x * C; gC += gR[0][1] * x * y; gz -= gR[0][1] * sa; gsa -= gR[0][1] * z;
  // R02 = z x C + y sa
  gz += gR[0][2] * x * C; gx += gR[0][2] * z * C; gC += gR[0][2] * z * x; gy += gR[0][2] * sa; gsa += gR[0][2] * y;
  // R10 = x y C + z sa
  gx += gR[1][0] * y * C; gy += gR[1][0] * x * C; gC += gR[1][0] * x * y; gz += gR[1][0] * sa; gsa += gR[1][0] * z;
  // R11 = y y C + ca
  gy += gR[1][1] * 2 * y * C; gC += gR[1][1] * y * y; gca += gR[1][1];
  // R12 = y z C - x sa
  gy += gR[1][2] * z * C; gz += gR[1][2] * y * C; gC += gR[1][2] * y * z; gx -= gR[1][2] * sa; gsa -= gR[1][2] * x;
  // R20 = z x C - y sa
  gz += gR[2][0] * x * C; gx += gR[2][0] * z * C; gC += gR[2][0] * z * x; gy -= gR[2][0] * sa; gsa -= gR[2][0] * y;
  // R21 = y z C + x sa
  gy += gR[2][1] * z * C; gz += gR[2][1] * y * C; gC += gR[2][1] * y * z; gx += gR[2][1] * sa; gsa += gR[2][1] * x;
  // R22 = z z C + ca
  gz += gR[2][2] * 2 * z * C; gC += gR[2][2] * z * z; gca += gR[2][2];
  gca -= gC;                                   // C = 1 - ca
  float gang = -r.sa * gca + r.ca * gsa;       // ca = cos(angle), sa = sin(angle)
  // axis = v / a, a = angle + 1e-7
  const float ga = -(gx * v[0] + gy * v[1] + gz * v[2]) / (r.a * r.a);
  gang += ga;
  float gv[3] = {gx / r.a, gy / r.a, gz / r.a};
  if (r.angle > 0.f)
    for (int k = 0; k < 3; ++k) gv[k] += gang * v[k] / r.angle;   // torch.norm backward (0 at the origin)
  for (int k = 0; k < 3; ++k) { gaa[k] = gv[k]; gtr[k] = gt[k]; }
}

// ------------------------------------------------------------------ small per-element pieces
// proj table: M = (K T)[:3,:3] * invK[:3,:3], p4 = (K T)[:3,3], in double then rounded once.
// value at fine pixel (y, x) of plane `d` (Hs x Ws, level s) up-sampled bilinearly to (Hs << s, Ws << s):
// F.interpolate(..., mode="bilinear", align_corners=False) (trainer.py:350-351, 451-454), torch upsample_bilinear2d
MD2_HD float upsample_at(const float* d, int lv, int Hs, int Ws, int y, int x) {
  if (lv == 0) return MD2_LD(d + y * Ws + x);
  const float rs = 1.0f / (float)(1 << lv);
  float sy = fmaf(rs, (float)y + 0.5f, -0.5f);
  sy = sy < 0.0f ? 0.0f : sy;
  float sx = fmaf(rs, (float)x + 0.5f, -0.5f);
  sx = sx < 0.0f ? 0.0f : sx;
  const int y0 = (int)sy, x0 = (int)sx;
  const int y1 = y0 + ((y0 < Hs - 1) ? 1 : 0), x1 = x0 + ((x0 < Ws - 1) ? 1 : 0);
  const float ly1 = sy - (float)y0, ly0 = 1.0f - ly1, lx1 = sx - (float)x0, lx0 = 1.0f - lx1;
  const float top = lx0 * MD2_LD(d + y0 * Ws + x0) + lx1 * MD2_LD(d + y0 * Ws + x1);
  const float bot = lx0 * MD2_LD(d + y1 * Ws + x0) + lx1 * MD2_LD(d + y1 * Ws + x1);
  return ly0 * top + ly1 * bot;
}

// posecnn (trainer.py:366-375): mean_inv_depth = (1 / depth).mean(3).mean(2) = a + c * mean(up-sampled disp_s);
// the sums come from acc_updisp (md2_updisp_sum)
MD2_HD void posecnn_mid(const Params& P, int s, int b) {
  const double m = P.acc[acc_updisp(P, s, b)] / ((double)P.H * P.W);
  P.mid[s * P.B + b] = (float)((double)P.a_disp + (double)P.c_disp * m);
}

// ps: pose set (scale under posecnn, else 0)
MD2_HD void setup_projection(const Params& P, int ps, int b, int f) {
  const float* K = P.K + (size_t)b * 16;
  float Tl[16];
  const float* T;
  if (P.aa[f]) {     // T from the pose leaves
    const float* aa = P.aa[f] + (size_t)b * P.pose_stride[f];
    const float* tr = P.tr[f] + (size_t)b * P.pose_stride[f];
    // the unscaled T is what predict_poses stores as outputs[("cam_T_cam", 0, f)] (trainer.py:294-295)
    if (ps == 0) pose_to_matrix(aa, tr, P.pose_invert[f], P.Tws[f] + (size_t)b * 16);
    if (P.posecnn) {
      const float m = P.mid[ps * P.B + b];
      const float trs[3] = {MD2_LD(tr) * m, MD2_LD(tr + 1) * m, MD2_LD(tr + 2) * m};     // trainer.py:374-375
      pose_to_matrix(aa, trs, P.pose_invert[f], Tl);
      T = Tl;
    } else {
      T = P.Tws[f] + (size_t)b * 16;
    }
  } else {
    T = P.Tm[f] + (size_t)b * 16;
  }
  const float* iK = P.invK + (size_t)b * 16;
  double Pm[3][4];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 4; ++j) {
      double a = 0.0;
      for (int k = 0; k < 4; ++k) a += (double)MD2_LD(K + i * 4 + k) * (double)T[k * 4 + j];   // (T may be the local Tl)
      Pm[i][j] = a;
    }
  float* o = P.proj + (size_t)((ps * P.B + b) * P.nsrc + f) * 12;
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) {
      double a = 0.0;
      for (int k = 0; k < 3; ++k) a += Pm[i][k] * (double)MD2_LD(iK + k * 4 + j);
      o[i * 3 + j] = (float)a;
    }
    o[9 + i] = (float)Pm[i][3];
  }
}

// Edge-aware smoothness at pixel (x,y) of scale s (layers.py:202-215 on the
// mean-normalised disparity of trainer.py:486-487).  Returns the pixel's two forward
// edge terms and gn = d(sum_x/Nx + sum_y/Ny) / d norm_disp(x,y).
MD2_HD float md2_exp_neg(float g) {
#if defined(__CUDA_ARCH__)
  return __expf(-g);
#else
  return expf(-g);
#endif
}
MD2_HD void smooth_pixel(const Params& P, int s, int b, int y, int x, float inv_m,
                         float& ex_out, float& ey_out, float& gn_out) {
  const int Hs = P.H >> P.lvl[s], Ws = P.W >> P.lvl[s];
  const size_t plane = (size_t)Hs * Ws;
  const float* d = P.disp[s] + (size_t)b * plane;
  const size_t p = (size_t)y * Ws + x;
  const float inx = 1.0f / ((float)P.B * (float)Hs * (float)(Ws - 1));
  const float iny = 1.0f / ((float)P.B * (float)(Hs - 1) * (float)Ws);
  const float n0 = MD2_LD(d + p) * inv_m;
  auto px = [&](int c, size_t q) { return load_px(P.color[s], P.color8[s], P.u8_hwc, b, c, (int)plane, (int)q); };
  const float i0 = px(0, p), i1 = px(1, p), i2 = px(2, p);
  float gn = 0.f, ex = 0.f, ey = 0.f;
  // one edge between this pixel and the neighbour at offset `o`; `fwd` = this pixel is the first end
  auto edge = [&](size_t q, bool fwd, float scale, float& e_out) {
    const float g = fabsf(i0 - px(0, q)) + fabsf(i1 - px(1, q)) + fabsf(i2 - px(2, q));
    const float w = md2_exp_neg(g * (1.0f / 3.0f));
    const float df = n0 - MD2_LD(d + q) * inv_m;          // n(this) - n(neighbour)
    MD2_DBG(if (fwd) {
      signed char* arr = (q == p + 1) ? D.smx : D.smy;
      arr[D.smoff[s] + (long)b * plane + (long)p] = (signed char)(df > 0.f ? 1 : (df < 0.f ? -1 : 0));
    });
    if (fwd) e_out = fabsf(df) * w;
    // d|n_a - n_b| / d n(this) = sign(n(this) - n(neighbour)) for either end of the edge
    gn += scale * ((df > 0.f) ? w : ((df < 0.f) ? -w : 0.f));
  };
  float dummy;
  if (x + 1 < Ws) edge(p + 1, true, inx, ex);
  if (x > 0) edge(p - 1, false, inx, dummy);
  if (y + 1 < Hs) edge(p + Ws, true, iny, ey);
  if (y > 0) edge(p - Ws, false, iny, dummy);
  ex_out = ex; ey_out = ey; gn_out = gn;
}

// Per-(scale, sample) scalars of the smoothness adjoint (A.4): 1/m and (sum gn*disp)/(m^2 N).
MD2_HD void smooth_scalars(const Params& P, int s, int b, float& inv_m, float& dterm) {
  const int n = (P.H >> P.lvl[s]) * (P.W >> P.lvl[s]);
  const float m = (float)(P.acc[acc_dispsum(P, s, b)] / (double)n) + 1e-7f;
  inv_m = 1.0f / m;
  dterm = (float)P.acc[acc_dot(P, s, b)] / (m * m * (float)n);
}
// Smoothness part of d loss / d disp_s at pixel p (A.4).
MD2_HD float final_smooth_grad(const Params& P, int s, int b, int p, float inv_m, float dterm) {
  const int n = (P.H >> P.lvl[s]) * (P.W >> P.lvl[s]);
  const float wsm = P.smooth_w[s] / (float)P.S;
  return wsm * (MD2_LD(P.gn[s] + (size_t)b * n + p) * inv_m - dterm);
}

// Adjoint of the bilinear up-sampling (trainer.py:350-351) in gather form: the share of coarse
// pixel (X,Y) of scale s contributed by the fine rows ylo+j, ylo+j+K, ... (j in [0,K), K = 2^s).
// The 2K x 2K fine pixels whose taps can hit (X,Y) are visited with the forward weights.
// Weight with which fine index K*X - K/2 + i (i in [0,2K)) feeds coarse index X under torch's
// bilinear up-sampling with align_corners=False (src = (x+0.5)/K - 0.5 clamped at 0, second tap
// clamped at n-1).  Interior: the triangle (i+0.5)/K | (2K-i-0.5)/K (all dyadic, exact in fp32);
// first / last coarse index: the clamped taps add up to 1, fine indices outside the image get 0.
template <int K>
MD2_HD float up_weight(int i, int X, int n) {
  const float tri = (i < K) ? ((float)i + 0.5f) * (1.0f / (float)K) : ((float)(2 * K - i) - 0.5f) * (1.0f / (float)K);
  if (X == 0 && i < K) return (i < K / 2) ? 0.0f : 1.0f;
  if (X == n - 1 && i >= K) return (i < K + K / 2) ? 1.0f : 0.0f;
  return tri;
}
template <int K>
MD2_HD float upsample_adjoint_part(const Params& P, int s, int b, int Y, int X, int j) {
  const int Hs = P.H >> P.lvl[s], Ws = P.W >> P.lvl[s];
  const float cst = P.posecnn ? MD2_LD(P.gmidc + s * P.B + b) : 0.0f;    // see final_pose_posecnn
  const float* dD = P.dD[s] + (size_t)b * P.H * P.W;
  const int xlo = K * X - K / 2, ylo = K * Y - K / 2;
  const bool interior_x = (X > 0) && (X < Ws - 1);
  float acc = 0.f;
#pragma unroll
  for (int ry = 0; ry < 2; ++ry) {
    const int iy = j + ry * K;
    const int y = ylo + iy;
    const float wy = up_weight<K>(iy, Y, Hs);
    const int yc = y < 0 ? 0 : (y >= P.H ? P.H - 1 : y);
    const float* rowp = dD + yc * P.W;
    float row = 0.f;
    if (interior_x) {
      // fast path: all 2K fine columns are inside the image, compile-time triangle weights
#pragma unroll
      for (int i = 0; i < 2 * K; ++i) {
        const float w = (i < K) ? ((float)i + 0.5f) * (1.0f / (float)K) : ((float)(2 * K - i) - 0.5f) * (1.0f / (float)K);
        row = fmaf(w, MD2_LD(rowp + xlo + i) + cst, row);
      }
    } else {
#pragma unroll
      for (int i = 0; i < 2 * K; ++i) {
        const int x = xlo + i;
        const int xc = x < 0 ? 0 : (x >= P.W ? P.W - 1 : x);
        row = fmaf(up_weight<K>(i, X, Ws), MD2_LD(rowp + xc) + cst, row);
      }
    }
    acc = fmaf(wy, row, acc);
  }
  return acc;
}

// Scalar epilogue: losses and d loss / d cam_T_cam = K[:3,:]^T dP  (A.3).
MD2_HD void final_scalars(const Params& P) {
  double total = 0.0;
  for (int s = 0; s < P.S; ++s) {
    const int Hs = P.H >> P.lvl[s], Ws = P.W >> P.lvl[s];
    const double photo = P.acc[acc_photo(s)] / ((double)P.B * P.H * P.W);
    double sx = 0.0, sy = 0.0;
    for (int b = 0; b < P.B; ++b) { sx += P.acc[acc_smx(P, s, b)]; sy += P.acc[acc_smy(P, s, b)]; }
    const double sm = sx / ((double)P.B * Hs * (Ws - 1)) + sy / ((double)P.B * (Hs - 1) * Ws);
    double ls = photo + (double)P.smooth_w[s] * sm;
    if (P.pmask_on)       // trainer.py:458-459: loss += 0.2 * BCELoss(mask, ones)
      ls += 0.2 * P.acc[acc_bce(P, s)] / ((double)P.B * P.nsrc * P.H * P.W);
    P.losses[1 + s] = (float)ls;
    total += ls;
  }
  P.losses[0] = (float)(total / P.S);
}
MD2_HD void final_grad_T(const Params& P, int b, int f) {
  if (P.posecnn) return;            // see final_pose_posecnn
  float* g = P.grad_T[f];
  const bool leaves = P.aa[f] && P.grad_aa[f] && P.grad_tr[f];
  if (!g && !leaves) return;
  const float* K = P.K + (size_t)b * 16;
  float gT[16];
  for (int k = 0; k < 4; ++k)
    for (int j = 0; j < 4; ++j) {
      double a = 0.0;
      if (P.pose_grad[f])
        for (int i = 0; i < 3; ++i) a += (double)MD2_LD(K + i * 4 + k) * P.acc[acc_dP(P, 0, b, f, i * 4 + j)];
      gT[k * 4 + j] = (float)(a * (double)P.gscale);
    }
  if (g)
    for (int i = 0; i < 16; ++i) g[(size_t)b * 16 + i] = gT[i];
  if (leaves)      // adjoint of transformation_from_parameters: the pose gradient leaves the path here
    pose_to_matrix_backward(gT, P.aa[f] + (size_t)b * P.pose_stride[f], P.tr[f] + (size_t)b * P.pose_stride[f],
                            P.pose_invert[f], P.grad_aa[f] + (size_t)b * 3, P.grad_tr[f] + (size_t)b * 3);
}

// posecnn epilogue of sample b: the pose gradient of every scale flows through transformation_from_parameters
// (layers.py:28-45) to the leaves - axisangle directly, translation through the factor mean_inv_depth (trainer.py:374-375)
// - and through that factor to every pixel of the up-sampled disparity of the scale (gmidc, added by the final pass).
MD2_HD void final_pose_posecnn(const Params& P, int b) {
  const float* K = P.K + (size_t)b * 16;
  float gaa[kMaxSrc][3], gtr[kMaxSrc][3];
  for (int f = 0; f < P.nsrc; ++f)
    for (int i = 0; i < 3; ++i) { gaa[f][i] = 0.f; gtr[f][i] = 0.f; }
  for (int ps = 0; ps < P.S; ++ps) {
    const float m = P.mid[ps * P.B + b];
    float gm = 0.f;
    for (int f = 0; f < P.nsrc; ++f) {
      if (!P.aa[f] || !P.pose_grad[f]) continue;
      float gT[16];
      for (int k = 0; k < 4; ++k)
        for (int j = 0; j < 4; ++j) {
          double a = 0.0;
          for (int i = 0; i < 3; ++i) a += (double)MD2_LD(K + i * 4 + k) * P.acc[acc_dP(P, ps, b, f, i * 4 + j)];
          gT[k * 4 + j] = (float)(a * (double)P.gscale);
        }
      const float* aa = P.aa[f] + (size_t)b * P.pose_stride[f];
      const float* tr = P.tr[f] + (size_t)b * P.pose_stride[f];
      const float trs[3] = {MD2_LD(tr) * m, MD2_LD(tr + 1) * m, MD2_LD(tr + 2) * m};
      float ga[3], gt[3];
      pose_to_matrix_backward(gT, aa, trs, P.pose_invert[f], ga, gt);
      for (int i = 0; i < 3; ++i) {
        gaa[f][i] += ga[i];
        gtr[f][i] = fmaf(gt[i], m, gtr[f][i]);
        gm = fmaf(gt[i], MD2_LD(tr + i), gm);
      }
    }
    // d mean_inv_depth / d (up-sampled disp)(p) = c / (H W)
    P.gmidc[ps * P.B + b] = (float)((double)gm * (double)P.c_disp / ((double)P.H * P.W));
  }
  for (int f = 0; f < P.nsrc; ++f) {
    if (!P.aa[f]) continue;
    if (P.grad_aa[f]) for (int i = 0; i < 3; ++i) P.grad_aa[f][(size_t)b * 3 + i] = gaa[f][i];
    if (P.grad_tr[f]) for (int i = 0; i < 3; ++i) P.grad_tr[f][(size_t)b * 3 + i] = gtr[f][i];
  }
}

// --predictive_mask: pixel (y, x) of the mask of (scale s, sample b, source f) up-sampled to full resolution
// (trainer.py:451-454); stores it in the plane the marching pass reads and returns its BCE term against 1
// (nn.BCELoss clamps log at -100, trainer.py:458)
MD2_HD float pmask_up_pixel(const Params& P, int s, int b, int f, int y, int x) {
  const int Hs = P.H >> P.lvl[s], Ws = P.W >> P.lvl[s];
  const float m = upsample_at(P.pmask[s] + (size_t)(b * P.nsrc + f) * Hs * Ws, P.lvl[s], Hs, Ws, y, x);
  P.pm[s][((size_t)(b * P.nsrc + f) * P.H + y) * P.W + x] = m;
  const float lg = logf(m);
  return -(lg < -100.0f ? -100.0f : lg);
}
// d loss / d (up-sampled mask) at full-resolution index i of the (b, f) plane: photometric part written by the
// marching pass + the BCE part (torch binary_cross_entropy_backward with target 1: (x - 1) / max((1 - x) x, 1e-12)),
// 0.2 / (B nsrc H W) per scale and 1 / S for the total
MD2_HD float pmask_full_grad(const Params& P, int s, size_t i) {
  const float m = MD2_LD(P.pm[s] + i);
  const float den = (1.0f - m) * m;
  const float bce = (m - 1.0f) / (den > 1e-12f ? den : 1e-12f);
  const float k = (float)(0.2 / ((double)P.B * P.nsrc * P.H * P.W * P.S));
  return MD2_LD(P.gpm[s] + i) + k * bce;
}
// adjoint of the up-sampling for the mask: coarse pixel (Y, X) of plane (b, f) at scale s, gather form
template <int K>
MD2_HD float pmask_adjoint(const Params& P, int s, int b, int f, int Y, int X) {
  const int Hs = P.H >> P.lvl[s], Ws = P.W >> P.lvl[s];
  const size_t base = (size_t)(b * P.nsrc + f) * P.H * P.W;
  if (K == 1) return pmask_full_grad(P, s, base + (size_t)Y * P.W + X);
  const int xlo = K * X - K / 2, ylo = K * Y - K / 2;
  float acc = 0.f;
  for (int iy = 0; iy < 2 * K; ++iy) {
    const int y = ylo + iy;
    const float wy = up_weight<K>(iy, Y, Hs);
    if (y < 0 || y >= P.H || wy == 0.0f) continue;
    float row = 0.f;
    for (int i = 0; i < 2 * K; ++i) {
      const int x = xlo + i;
      const float wx = up_weight<K>(i, X, Ws);
      if (x < 0 || x >= P.W || wx == 0.0f) continue;
      row = fmaf(wx, pmask_full_grad(P, s, base + (size_t)y * P.W + x), row);
    }
    acc = fmaf(wy, row, acc);
  }
  return acc;
}
MD2_HD void pmask_grad_pixel(const Params& P, int s, int b, int f, int Y, int X) {
  const int lv = (P.lvl4 >> (4 * s)) & 15;
  const int Hs = P.H >> lv, Ws = P.W >> lv;
  float g;
  switch (lv) {
    case 0: g = pmask_adjoint<1>(P, s, b, f, Y, X); break;
    case 1: g = pmask_adjoint<2>(P, s, b, f, Y, X); break;
    case 2: g = pmask_adjoint<4>(P, s, b, f, Y, X); break;
    default: g = pmask_adjoint<8>(P, s, b, f, Y, X); break;
  }
  P.grad_pmask[s][((size_t)(b * P.nsrc + f) * Hs + Y) * Ws + X] = g;
}

}  // namespace md2
