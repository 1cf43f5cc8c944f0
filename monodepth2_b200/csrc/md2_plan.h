// md2_plan.h - host-side planner: validates an md2_problem, lays out the workspace
// and fills the device-side Params block.  Shared by the CUDA C-ABI (md2_capi.cu) and
// by the host emulator used in tests (tests/emu/md2_emu.cpp).
#pragma once

#include <stddef.h>
#include <stdint.h>
#include <string.h>

#include "../../include/md2_loss.h"
#include "md2_core.cuh"

namespace md2 {

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Layout {
  size_t acc_off, acc_bytes;
  size_t proj_off, idloss_off, smsc_off;
  size_t tgt4_off, src4_off[kMaxSrc];
  size_t dD_off[kMaxScales], gn_off[kMaxScales], zup_off[kMaxScales];
  size_t Tws_off[kMaxSrc];
  size_t mid_off, gmidc_off;                       // posecnn
  size_t pm_off[kMaxScales], gpm_off[kMaxScales];  // predictive mask
  size_t cvt_img_off[1 + kMaxSrc], cvt_col_off[kMaxScales];   // uint8 entry: frames / pyramid as planar float
  size_t wd_disp_off[kMaxScales], wd_pm_off[kMaxScales];      // bf16 / fp16 leaves widened to fp32 (md2_widen)
  size_t wd_pose_off[kMaxSrc];                                // T (16 B floats) or axisangle | translation (3 B each)
  size_t total;
};

// bf16 / fp16 leaves (md2_problem::*_dtype): md2_widen copies each into an fp32 workspace buffer before the prologue,
// and the Params pointers are redirected to the copies, so no kernel downstream knows the leaves were narrower.
// Element i of a job reads src[(i / row) * stride + i % row] (row = 0: src[i]).
constexpr int kMaxWiden = 2 * kMaxScales + 2 * kMaxSrc;
struct WidenJob {
  const void* src;
  float* dst;
  long long n;
  int row, stride, dtype;
};
struct Widen {
  int n;                 // jobs; 0 = nothing to launch (every leaf fp32)
  long long max_n;       // largest job, sizes the grid
  WidenJob job[kMaxWiden];
};

// Pyramid level of scale slot s: md2_problem::scale_level when given (strictly ascending, trainer.py:345,413 iterate
// opt.scales; the dataloader builds levels 0..3 whatever --scales says, trainer.py:127-135), else s.
inline bool custom_levels(const md2_problem* p) {
  for (int s = 0; s < MD2_MAX_SCALES; ++s) if (p->scale_level[s] != 0) return true;
  return false;
}
inline int level_of(const md2_problem* p, int s) { return custom_levels(p) ? p->scale_level[s] : s; }

inline bool dtype_ok(int d) { return d == MD2_DTYPE_F32 || d == MD2_DTYPE_BF16 || d == MD2_DTYPE_F16; }

inline int validate(const md2_problem* p) {
  if (!p) return MD2_ERR_INVALID_ARGUMENT;
  if (!dtype_ok(p->disp_dtype) || !dtype_ok(p->pmask_dtype)) return MD2_ERR_INVALID_ARGUMENT;
  for (int f = 0; f < MD2_MAX_SRC; ++f) if (!dtype_ok(p->pose_dtype[f])) return MD2_ERR_INVALID_ARGUMENT;
  if (p->batch < 1 || p->height < 4 || p->width < 4) return MD2_ERR_INVALID_ARGUMENT;
  if (p->num_scales < 1 || p->num_scales > MD2_MAX_SCALES) return MD2_ERR_INVALID_ARGUMENT;
  if (p->num_src < 1 || p->num_src > MD2_MAX_SRC) return MD2_ERR_INVALID_ARGUMENT;
  for (int s = 0; s < p->num_scales; ++s) {
    const int lv = level_of(p, s);
    if (lv < 0 || lv >= MD2_MAX_SCALES) return MD2_ERR_INVALID_ARGUMENT;
    if (s > 0 && lv <= level_of(p, s - 1)) return MD2_ERR_INVALID_ARGUMENT;     // ascending, no duplicates
  }
  // level 0 is part of every list the reference accepts: it warps at source_scale 0 with backproject_depth[0] /
  // project_3d[0], which it builds for opt.scales only (trainer.py:151-159,377)
  if (level_of(p, 0) != 0) return MD2_ERR_INVALID_ARGUMENT;
  const int top = level_of(p, p->num_scales - 1);
  const int div = 1 << top;
  if (p->height % div || p->width % div) return MD2_ERR_INVALID_ARGUMENT;
  if ((p->height >> top) < 2 || (p->width >> top) < 2) return MD2_ERR_INVALID_ARGUMENT;
  if (!(p->min_depth > 0.f) || !(p->max_depth > p->min_depth)) return MD2_ERR_INVALID_ARGUMENT;
  if ((long long)p->batch * 3 * p->height * p->width * MD2_MAX_SRC >= (1LL << 31)) return MD2_ERR_UNSUPPORTED;
  // trainer.py:90-92: "When using predictive_mask, please disable automasking with --disable_automasking"
  if (p->predictive_mask && p->automask) return MD2_ERR_INVALID_ARGUMENT;
  return MD2_OK;
}

inline Layout make_layout(const md2_problem* p) {
  Layout L;
  memset(&L, 0, sizeof(L));
  const size_t B = p->batch, H = p->height, W = p->width;
  size_t off = 0;
  const size_t npose = p->posecnn ? p->num_scales : 1;
  const size_t nacc = 3 * kMaxScales + 5 * kMaxScales * B + npose * B * p->num_src * 12 + kMaxScales;   // = acc_count()
  L.acc_off = off; L.acc_bytes = nacc * sizeof(double);
  off = align_up(off + L.acc_bytes, 256);
  L.proj_off = off; off = align_up(off + npose * B * p->num_src * 12 * sizeof(float), 256);
  L.mid_off = off; off = align_up(off + kMaxScales * B * sizeof(float), 256);
  L.gmidc_off = off; off = align_up(off + kMaxScales * B * sizeof(float), 256);
  L.smsc_off = off; off = align_up(off + kMaxScales * B * 2 * sizeof(float), 256);
  for (int f = 0; f < p->num_src; ++f) { L.Tws_off[f] = off; off = align_up(off + B * 16 * sizeof(float), 256); }
  L.idloss_off = off; off = align_up(off + B * p->num_src * H * W * sizeof(float), 256);
  L.tgt4_off = off; off = align_up(off + B * H * W * 4 * sizeof(float), 256);
  for (int f = 0; f < p->num_src; ++f) {
    L.src4_off[f] = off; off = align_up(off + B * H * W * 4 * sizeof(float), 256);
  }
  for (int s = 0; s < p->num_scales; ++s) {
    L.dD_off[s] = off; off = align_up(off + B * H * W * sizeof(float), 256);
    L.zup_off[s] = off; off = align_up(off + B * H * W * sizeof(float), 256);
    L.gn_off[s] = off; off = align_up(off + B * (H >> level_of(p, s)) * (W >> level_of(p, s)) * sizeof(float), 256);
    if (p->predictive_mask) {
      L.pm_off[s] = off; off = align_up(off + B * p->num_src * H * W * sizeof(float), 256);
      L.gpm_off[s] = off; off = align_up(off + B * p->num_src * H * W * sizeof(float), 256);
    }
  }
  // (reserved whether or not the caller uses the uint8 entry: the workspace size is a function of md2_problem alone)
  for (int i = 0; i <= p->num_src; ++i) { L.cvt_img_off[i] = off; off = align_up(off + B * 3 * H * W * sizeof(float), 256); }
  for (int s = 0; s < p->num_scales; ++s) {
    const int lv = level_of(p, s);
    if (lv == 0) continue;                      // level 0 = the converted target frame
    L.cvt_col_off[s] = off; off = align_up(off + B * 3 * (H >> lv) * (W >> lv) * sizeof(float), 256);
  }
  // fp32 copies of reduced-precision leaves, after everything else: an all-fp32 problem keeps its layout and size
  for (int s = 0; s < p->num_scales; ++s) {
    const int lv = level_of(p, s);
    const size_t plane = (H >> lv) * (W >> lv);
    if (p->disp_dtype != MD2_DTYPE_F32) { L.wd_disp_off[s] = off; off = align_up(off + B * plane * sizeof(float), 256); }
    if (p->predictive_mask && p->pmask_dtype != MD2_DTYPE_F32) {
      L.wd_pm_off[s] = off; off = align_up(off + B * p->num_src * plane * sizeof(float), 256);
    }
  }
  for (int f = 0; f < p->num_src; ++f)
    if (p->pose_dtype[f] != MD2_DTYPE_F32) { L.wd_pose_off[f] = off; off = align_up(off + B * 16 * sizeof(float), 256); }
  L.total = off;
  return L;
}

inline int default_seg_rows(const md2_problem* p) {
  // Rows marched per warp job.  A job marches r + 4 rows (2 halo rows each side) and the kernel runs in waves of
  // 148 SMs x 8 warps (12 for the forward-only instantiations): minimise waves x (r + 4) over r = ceil(H / n).
  // Measured on B200 (profiles/r01_optimization_log.md): 640x192 x 12: 96 rows 0.474 ms, 64 rows 0.480 ms,
  // 48 rows 0.486 ms per step; 1024x320: 160 rows 1.170 ms, 80 rows 1.185 ms, 107 rows 1.251 ms.
  // Round 2 (role-specialised kernel, one CTA per job, 5 CTAs per SM = 740 slots with gradients): the same model with
  // 740 slots picks the same heights (96 / 160), and the sweeps on the final kernel agree: 640x192 96 rows 0.3216 ms,
  // 64 rows 0.3252, 48 rows 0.3334, 192 rows 0.3444; 1024x320 160 rows 0.7955 ms, 107 rows 0.7988, 80 rows 0.8015.
  if (p->rows_per_segment > 0) return p->rows_per_segment < p->height ? p->rows_per_segment : p->height;
  const long slots = 148L * (p->want_grad ? 8 : 12);
  const long nband = (p->width + kOwnCols - 1) / kOwnCols;
  int best_r = p->height;
  long best_cost = -1;
  // (n = 1, one job per band, is excluded when the image is tall enough to split: measured 0.654 ms at 640x192
  // although the model rates it best - all warps then stream the same image rows in lock step)
  for (int n = (p->height >= 48 ? 2 : 1); n <= 8; ++n) {
    const int r = (p->height + n - 1) / n;
    if (n > 1 && r < 24) break;
    const long jobs = (long)p->num_scales * p->batch * nband * ((p->height + r - 1) / r);
    const long cost = ((jobs + slots - 1) / slots) * (r + 4);
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_r = r; }
  }
  return best_r;
}

// Fills `P`.  Returns MD2_OK or an error when required tensors are missing.
inline int fill_params(const md2_problem* p, const md2_tensors* t, void* workspace, Params* P) {
  if (!t || !workspace) return MD2_ERR_INVALID_ARGUMENT;
  memset(P, 0, sizeof(*P));
  const Layout L = make_layout(p);
  char* ws = (char*)workspace;
  P->B = p->batch; P->H = p->height; P->W = p->width; P->S = p->num_scales; P->nsrc = p->num_src;
  P->automask = p->automask ? 1 : 0;
  P->avg = p->avg_reprojection ? 1 : 0;
  P->nid = P->automask ? (P->avg ? 1 : P->nsrc) : 0;
  P->align_corners = p->align_corners ? 1 : 0;
  P->want_grad = p->want_grad ? 1 : 0;
  P->no_ssim = p->no_ssim ? 1 : 0;
  P->posecnn = p->posecnn ? 1 : 0;
  P->npose = P->posecnn ? p->num_scales : 1;
  P->pmask_on = p->predictive_mask ? 1 : 0;
  // layers.py:21-23: min_disp = 1/max_depth, max_disp = 1/min_depth (python doubles -> fp32 scalars)
  const double lo = 1.0 / (double)p->max_depth, hi = 1.0 / (double)p->min_depth;
  P->a_disp = (float)lo;
  P->c_disp = (float)(hi - lo);
  const double W = p->width, H = p->height;
  if (P->align_corners) { P->sx = 1.f; P->ox = 0.f; P->sy = 1.f; P->oy = 0.f; }
  else {
    // layers.py:190-192 then grid_sample un-normalisation with align_corners=False:
    // ix = ((u/(W-1) - 0.5)*2 + 1) * W/2 - 0.5 = u*W/(W-1) - 0.5
    P->sx = (float)(W / (W - 1.0)); P->ox = -0.5f;
    P->sy = (float)(H / (H - 1.0)); P->oy = -0.5f;
  }
  P->wmax = (float)(p->width - 1); P->hmax = (float)(p->height - 1);
  P->eps = 1e-7f;
  P->gscale = (float)(1.0 / ((double)p->num_scales * p->batch * H * W) / (P->avg ? (double)p->num_src : 1.0));
  for (int s = 0; s < p->num_scales; ++s) {
    P->lvl[s] = level_of(p, s);
    P->smooth_w[s] = (float)((double)p->disparity_smoothness / (double)(1 << P->lvl[s]));   // trainer.py:491: / (2 ** scale)
  }
  P->up0 = P->lvl[0] == 0 ? 1 : 0;
  for (int s = 0; s < p->num_scales; ++s) P->lvl4 |= P->lvl[s] << (4 * s);
  P->noise_event = t->noise_ready_event;
  P->seg_rows = default_seg_rows(p);
  P->nseg = (p->height + P->seg_rows - 1) / P->seg_rows;
  P->nband = (p->width + kOwnCols - 1) / kOwnCols;
  P->nband_id = (p->width + kIdCols - 1) / kIdCols;
  // the identity pass runs 16 warps per SM (<= 128 registers): pick the segment height that minimises
  // (waves of 148 SMs x 16 warps) x (rows marched per job, 2 of them halo) - e.g. 24 rows at 640x192 x 12
  // (one 89 %-full wave of 26 rows instead of two waves of 18); measured: whole step 0.496 -> 0.489 ms at
  // 640x192, 1.225 -> 1.203 ms at 1024x320
  {
    const long slots = 148L * 16;
    int best_r = p->height < 16 ? p->height : 16;
    long best_cost = -1;
    const int rmax = p->height < 64 ? p->height : 64;
    for (int r = 8; r <= rmax; ++r) {
      const long jobs = (long)p->batch * P->nband_id * ((p->height + r - 1) / r);
      const long cost = ((jobs + slots - 1) / slots) * (r + 2);
      if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_r = r; }
    }
    P->id_rows = best_r;
  }
  P->nseg_id = (p->height + P->id_rows - 1) / P->id_rows;
  const bool u8 = t->target_u8 != nullptr;
  if ((!u8 && !t->target) || !t->K || !t->inv_K || !t->losses) return MD2_ERR_INVALID_ARGUMENT;
  P->tgt = u8 ? nullptr : t->target; P->K = t->K; P->invK = t->inv_K;
  P->tgt8 = t->target_u8; P->u8_hwc = t->u8_hwc ? 1 : 0;
  for (int f = 0; f < p->num_src; ++f) {
    if (u8 ? !t->source_u8[f] : !t->source[f]) return MD2_ERR_INVALID_ARGUMENT;
    if (t->axisangle[f]) {          // T built in the call from the pose leaves
      if (!t->translation[f] || t->pose_stride[f] < 3) return MD2_ERR_INVALID_ARGUMENT;
      P->aa[f] = t->axisangle[f]; P->tr[f] = t->translation[f];
      P->pose_stride[f] = t->pose_stride[f]; P->pose_invert[f] = t->pose_invert[f] ? 1 : 0;
      P->Tws[f] = t->cam_T_cam[f] ? t->cam_T_cam[f] : (float*)(ws + L.Tws_off[f]);
      P->Tm[f] = P->Tws[f];
      if (p->want_grad && t->pose_requires_grad[f]) {
        if (!t->grad_axisangle[f] || !t->grad_translation[f]) return MD2_ERR_INVALID_ARGUMENT;
        P->grad_aa[f] = t->grad_axisangle[f]; P->grad_tr[f] = t->grad_translation[f];
      }
    } else {
      if (!t->T[f]) return MD2_ERR_INVALID_ARGUMENT;
      P->Tm[f] = t->T[f];
      // posecnn: a source given as a fixed matrix keeps that matrix at every scale and gets no pose gradient
      if (p->posecnn && t->pose_requires_grad[f] && p->want_grad) return MD2_ERR_INVALID_ARGUMENT;
    }
    P->src[f] = u8 ? nullptr : t->source[f];
    P->src8[f] = u8 ? t->source_u8[f] : nullptr;
    P->pose_grad[f] = (t->pose_requires_grad[f] && p->want_grad) ? 1 : 0;
    // posecnn: the disparity gradient depends on the pose adjoint (through mean_inv_depth) whether or not the leaves
    // themselves want one
    if (p->posecnn && p->want_grad && t->axisangle[f]) P->pose_grad[f] = 1;
    P->grad_T[f] = p->want_grad ? t->grad_T[f] : nullptr;
  }
  for (int s = 0; s < p->num_scales; ++s) {
    const unsigned char* c8 = u8 ? (t->color_u8[s] ? t->color_u8[s] : (P->lvl[s] == 0 ? t->target_u8 : nullptr)) : nullptr;
    if (!t->disp[s] || (u8 ? !c8 : !t->color[s])) return MD2_ERR_INVALID_ARGUMENT;
    if (P->automask && !t->noise[s]) return MD2_ERR_INVALID_ARGUMENT;
    if (p->want_grad && !t->grad_disp[s]) return MD2_ERR_INVALID_ARGUMENT;
    P->disp[s] = t->disp[s]; P->color[s] = u8 ? nullptr : t->color[s]; P->color8[s] = c8; P->noise[s] = t->noise[s];
    P->grad_disp[s] = t->grad_disp[s];
    P->depth[s] = t->depth[s];
    P->idsel[s] = t->identity_selection[s];
    for (int f = 0; f < p->num_src; ++f) P->warped[f][s] = t->warped[f][s];
    P->dD[s] = t->grad_depth_dbg[s] ? t->grad_depth_dbg[s] : (float*)(ws + L.dD_off[s]);
    P->zup[s] = (float*)(ws + L.zup_off[s]);
    P->gn[s] = (float*)(ws + L.gn_off[s]);
    if (p->predictive_mask) {
      if (!t->pmask[s]) return MD2_ERR_INVALID_ARGUMENT;
      P->pmask[s] = t->pmask[s];
      P->pm[s] = (float*)(ws + L.pm_off[s]);
      P->gpm[s] = (float*)(ws + L.gpm_off[s]);
      P->grad_pmask[s] = p->want_grad ? t->grad_pmask[s] : nullptr;
    }
  }
  P->losses = t->losses;
  P->acc = (double*)(ws + L.acc_off);
  P->proj = (float*)(ws + L.proj_off);
  P->idloss = (float*)(ws + L.idloss_off);
  P->smsc = (float*)(ws + L.smsc_off);
  for (int i = 0; i <= p->num_src; ++i) P->cvt_img[i] = (float*)(ws + L.cvt_img_off[i]);
  for (int s = P->up0; s < p->num_scales; ++s) P->cvt_col[s] = (float*)(ws + L.cvt_col_off[s]);
  P->mid = (float*)(ws + L.mid_off);
  P->gmidc = (float*)(ws + L.gmidc_off);
  P->tgt4 = (float*)(ws + L.tgt4_off);
  for (int f = 0; f < p->num_src; ++f) P->src4[f] = (float*)(ws + L.src4_off[f]);
  return MD2_OK;
}

// After fill_params: lists the reduced-precision leaves in `Wd` and points `P` at their fp32 workspace copies.
inline void fill_widen(const md2_problem* p, void* workspace, Params* P, Widen* Wd) {
  memset(Wd, 0, sizeof(*Wd));
  const Layout L = make_layout(p);
  char* ws = (char*)workspace;
  auto add = [&](const void* src, size_t off, long long n, int row, int stride, int dtype) -> float* {
    WidenJob& j = Wd->job[Wd->n++];
    j.src = src; j.dst = (float*)(ws + off); j.n = n; j.row = row; j.stride = stride; j.dtype = dtype;
    if (n > Wd->max_n) Wd->max_n = n;
    return j.dst;
  };
  const long long B = p->batch;
  for (int s = 0; s < p->num_scales; ++s) {
    const long long plane = (long long)(p->height >> P->lvl[s]) * (p->width >> P->lvl[s]);
    if (p->disp_dtype != MD2_DTYPE_F32) P->disp[s] = add(P->disp[s], L.wd_disp_off[s], B * plane, 0, 0, p->disp_dtype);
    if (P->pmask_on && p->pmask_dtype != MD2_DTYPE_F32)
      P->pmask[s] = add(P->pmask[s], L.wd_pm_off[s], B * p->num_src * plane, 0, 0, p->pmask_dtype);
  }
  for (int f = 0; f < p->num_src; ++f) {
    const int d = p->pose_dtype[f];
    if (d == MD2_DTYPE_F32) continue;
    if (P->aa[f]) {         // pose leaves: 3 values per sample, pose_stride apart; the copies are packed (stride 3)
      P->aa[f] = add(P->aa[f], L.wd_pose_off[f], 3 * B, 3, P->pose_stride[f], d);
      P->tr[f] = add(P->tr[f], L.wd_pose_off[f] + 3 * B * sizeof(float), 3 * B, 3, P->pose_stride[f], d);
      P->pose_stride[f] = 3;
    } else {
      P->Tm[f] = add(P->Tm[f], L.wd_pose_off[f], 16 * B, 0, 0, d);
    }
  }
}

}  // namespace md2
