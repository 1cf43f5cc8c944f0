// md2_roles.cuh - the marching kernel, role-specialised (the default since round 2).
//
// The round-1 kernel kept the whole fused forward + adjoint state of a pixel column in one thread: ~240 registers,
// 8 warps per SM, and every warp ran one long dependent instruction stream per image row (measured: a warp alone
// needs ~3 250 cycles per row for 1 183 instructions; the kernel is bound by that latency, not by issue slots or
// bandwidth).
//
// Here the same per-lane arithmetic (md2_core.cuh / md2_pack2.cuh, unchanged) is split over warps that
// work on the SAME band of 32 columns, a few image rows apart, and hand rows to each other through
// shared memory:
//   role A  stage_a_issue + stage_a_finish of row t      (disparity -> depth -> projection -> gather ->
//           interpolation); publishes the row (target, pred, d pred / d (ix,iy), u, v, z) in a ring.
//   role B  stage_b of row t-1   (window sums, SSIM + L1, per-pixel minimum / automask, loss, the
//           SSIM-adjoint coefficients of the winner); reads its own and its neighbours' row from the
//           ring (no shuffles), publishes coefficients + winner in a second ring; its streamed inputs
//           (identity loss, tie-break noise) are loaded two rows ahead
//   role C  stage_c of row t-2   (3x3 box adjoint, d loss / d pred, grid-sample and projection
//           adjoints, d loss / d disparity, pose sums)
// One CTA = one band, one warp per role, one bar.sync per image row.  Each warp carries only its own role's rolling
// state (126-168 registers instead of 240-255, no spills with 1-3 sources), so 16 warps are resident per
// SM instead of 8, and the dependent chains of a row run concurrently on different warps instead of back
// to back in one.
//
// The forms that were measured and rejected (several role-A warps, cp.async gathers, the packed role C, the depth
// hand-over from role C, mbarrier-decoupled and free-running roles, ...) are recorded in profiles/r02_optimization_log.md.
#pragma once

#include "md2_core.cuh"
#include "md2_pack2.cuh"

namespace md2 {

// Measured on B200 (mono 640x192 x 12, md2_march_roles alone, profiles/r02_optimization_log.md):
//   1 A warp, 5 CTAs per SM (126 registers)  0.366 ms      2 A warps, 4 CTAs (128 registers)  0.402 ms
//   1 A warp, 4 CTAs (150 registers)         0.430 ms      3 A warps, 3 CTAs                  0.498 ms
//   1 A warp + cp.async gather, 5 CTAs       0.388 ms      round-1 kernel (one warp per band) 0.419 ms

// the role kernel keeps the backward box sums of every source count in registers (role C has room)
template <class C0>
struct RoleOf : C0 {
  static constexpr bool BSMEM = false;
  static constexpr bool ZUP = true;      // depth planes from md2_depth_up (see Cfg::ZUP)
  // branch-free stages B / C also under --avg_reprojection (measured at 640x192 x 12: 0.442 -> 0.413 ms; the two-source
  // per-pixel-minimum kernels lose with it: mono 0.326 -> 0.339 ms, --disable_automasking 0.358 -> 0.375 ms)
  static constexpr bool STRAIGHT = C0::STRAIGHT || C0::AVG;
};
// loops of the roles without a branch around the row body (the first / last periods, in which a role only crosses the
// barrier, are peeled): with the branch ptxas may park the wait for the loads a role keeps in flight across the barrier
// on that branch, at the top of the loop, instead of at their first use (measured: 29 % of role B's time)
// (one instantiation - 3 sources, --disable_automasking, SSIM, gradients - spills 12 bytes at its 168-register cap in
// the peeled form and keeps the branchy loops)
template <class C>
__host__ __device__ constexpr bool role_peel() {
  return !(C::NSRC == 3 && !C::AUTOMASK && C::GRAD && !C::AVG && !C::NOSSIM);
}
// the packed two-source role kernel runs its roles over PairedOf<C>: ring layout in the register pairs role B reads
// (see Cfg::PAIRED)
template <class C0>
struct PairedOf : C0 {
  static constexpr bool PAIRED = true;
};

template <class C>
struct RoleCfg {
  static constexpr int NA = 1;                                   // warps of role A (warp 0), then B, then C
  static constexpr int NROLES = NA + (C::GRAD ? 2 : 1);
  static constexpr int THREADS = 32 * NROLES;
  static constexpr int RING = C::GRAD ? 5 : 2;                   // rows in flight: A writes t, B reads t-1, C reads t-4
  // register budget per instantiation (no spills anywhere): 4 sources 255, 3 sources or --avg_reprojection with
  // gradients 168 (4 CTAs per SM: the 3-source kernel at 176 registers dropped to 3 CTAs and 0.81 ms instead of
  // 0.53 ms at 640x192 x 12), both together 224, everything else 136 (5 CTAs per SM)
  static constexpr int MIN_CTAS = (C::NSRC >= 4) ? 2 : (C::NSRC >= 3 && C::AVG && C::GRAD) ? 3 : ((C::NSRC >= 3 || C::AVG) && C::GRAD) ? 4 : 5;
  // registers per thread such that MIN_CTAS CTAs fit an SM (64 K registers, allocation unit 8 per thread); given as
  // __maxnreg__ rather than as the min-blocks argument of __launch_bounds__, under which ptxas picks 168 registers
  // plus a few bytes of spills for the 3-source kernels although 224 would fit
  // NOTE (5 CTAs of 96 threads): the arithmetic says 136, but a kernel that really USES 129-136 registers is given 4 CTAs
  // per SM (ncu launch__occupancy_limit_registers, measured on md2_march_mb: 0.43 instead of 0.33 ms).  Every shipped
  // 5-CTA instantiation uses <= 128 under this cap (tests/test_capi_symbols.py::test_register_budget reads the ptxas
  // log); capping at 128 instead makes ptxas schedule role B 6 instructions longer (0.329 vs 0.324 ms).
  static constexpr int MAXREG = ((65536 / (MIN_CTAS * THREADS)) / 8) * 8 > 255 ? 255 : ((65536 / (MIN_CTAS * THREADS)) / 8) * 8;
  static constexpr int NCF4 = (9 * C::NCS + 1 + 3) / 4;          // coefficient sets + winner tag, 16-byte fields
  static constexpr int STASH_F4 = RING * C::STASH4 * 32;
  static constexpr int COEF_F4 = C::GRAD ? 2 * NCF4 * 32 : 0;
  static constexpr int BAR_F4 = (RING * 8 + 15) / 16;            // one mbarrier per ring slot (TMA-staged target row)
  // + 19 unused 16-byte fields: the request every timing of this kernel was taken with.  Without them the request of
  // some 1- and 3-source instantiations falls below a carve-out step, and the driver may pick another L1 / shared split.
  static constexpr int SMEM_F4 = STASH_F4 + COEF_F4 + BAR_F4 + 19;
};

template <int NT>
__device__ __forceinline__ void role_sync() {
  asm volatile("bar.sync 0, %0;" ::"r"(NT) : "memory");
}

// Interior bands (WarpJob::staged): the 32 RGBx target texels of row t are one contiguous 512-byte run of the
// texel array and field 0 of a ring slot is one contiguous 512-byte run of shared memory, so the row is staged by a
// single TMA bulk copy (cp.async.bulk, UBLKCP) issued by one lane; its completion is tracked by the slot's mbarrier,
// which roles B and C wait on before they read the field.  No lane loads or stores the target.
// Kernels with gradients: role C issues the copy, right after its last read of the ring slot the row goes to, one
// period before role A fills the rest of that slot (role A is the role every barrier waits for, role C has ~50 %
// slack: profiles/r02f_march_roles.txt).  Forward-only kernels (no role C): role A, in the period of the row.
template <class C, class ST>
__device__ __forceinline__ void stage_target_row(const WarpJob& J, const ST& st, int t, int lane) {
  if (J.staged && lane == 0) {
    const int tr = reflect_clamp(t, J.H);
    const int slot = st.slot(t);
    mbar_expect_tx(st.tbar + slot, 32 * 16);
    tma_bulk_g2s(&st.at(slot, 0, C::STASH4), J.tgt4 + 4 * (tr * J.W + J.x0 - 2), 32 * 16, st.tbar + slot);
  }
}
// role C, period i (after its reads of slot(t0 + i - 4) == slot(t0 + i + 1)): stage the target row role A publishes next
template <class C, class ST>
__device__ __forceinline__ void stage_next_target_row(const WarpJob& J, const ST& st, int t, int t1, int lane) {
  if (C::GRAD && J.staged && t <= t1) {
    __syncwarp();
    stage_target_row<C>(J, st, t, lane);
  }
}
template <class C, class ST>
__device__ __forceinline__ void wait_target_row(const WarpJob& J, const ST& st, int t) {
  if (J.staged && t >= st.t0) mbar_wait(st.tbar + st.slot(t), st.parity(t));     // (rows before t0 are never staged)
}

// ---- role A: rows t0 .. t1, row t in the ring before the barrier that ends period (t - t0)
template <class C, class ST>
__device__ __forceinline__ void role_a(const Params& P, const WarpJob& J, int lane, const ST& st, int t0, int t1, int nit) {
  Lane<C> L;
  lane_init(L, P, J, lane);
  if (role_peel<C>()) {
#pragma unroll 1
    for (int t = t0; t <= t1; ++t) {
      if (!C::GRAD) stage_target_row<C>(J, st, t, lane);
      stage_a_issue<C, false, 1, true>(L, P, J, t);
      stage_a_finish<C, ST, true>(L, P, J, t, st);
      role_sync<RoleCfg<C>::THREADS>();
    }
#pragma unroll 1
    for (int p = t1 - t0 + 1; p < nit; ++p) role_sync<RoleCfg<C>::THREADS>();
    return;
  }
#pragma unroll 1
  for (int p = 0; p < nit; ++p) {
    const int t = t0 + p;
    if (t <= t1) {
      if (!C::GRAD) stage_target_row<C>(J, st, t, lane);
      stage_a_issue<C, false, 1, true>(L, P, J, t);
      stage_a_finish<C, ST, true>(L, P, J, t, st);
    }
    role_sync<RoleCfg<C>::THREADS>();
  }
}

// ---- role B, one row: reads its own and its neighbours' row t from the ring, stage_b, publishes the
// coefficients + winner into the 16-byte fields at `o`
template <class C, class ST>
__device__ __forceinline__ void b_step(Lane<C>& L, const Params& P, const WarpJob& J, int lane, const ST& st, F4* o,
                                       int t, int ol, int orr) {
  typedef RoleCfg<C> RC;
  const int slot = st.slot(t);
  Xchg1<C> lf, rt;
  wait_target_row<C>(J, st, t);
  {
    const F4* p = &st.at(slot, 0, C::STASH4);
    const F4 c = p[0], l = p[ol], r = p[orr];
    L.tg[0] = c.x; L.tg[1] = c.y; L.tg[2] = c.z;
    lf.tg[0] = l.x; lf.tg[1] = l.y; lf.tg[2] = l.z;
    rt.tg[0] = r.x; rt.tg[1] = r.y; rt.tg[2] = r.z;
  }
#pragma unroll
  for (int f = 0; f < C::NSRC; ++f) {
    const F4* p = &st.at(slot, 1 + 3 * f, C::STASH4);
    const F4 c = p[0], l = p[ol], r = p[orr];
    L.pr[f][0] = c.x; L.pr[f][1] = c.y; L.pr[f][2] = c.z;
    lf.pr[f][0] = l.x; lf.pr[f][1] = l.y; lf.pr[f][2] = l.z;
    rt.pr[f][0] = r.x; rt.pr[f][1] = r.y; rt.pr[f][2] = r.z;
  }
  stage_b(L, P, J, t, lane, lf, rt);
  if (C::GRAD) {
    float v[4 * RC::NCF4];
#pragma unroll
    for (int k = 0; k < 4 * RC::NCF4; ++k) v[k] = 0.f;
#pragma unroll
    for (int n = 0; n < C::NCS; ++n)
#pragma unroll
      for (int k = 0; k < 9; ++k) v[n * 9 + k] = L.coef[n][k];
    v[9 * C::NCS] = __int_as_float(L.tag);
#pragma unroll
    for (int k = 0; k < RC::NCF4; ++k) o[k * 32] = make_f4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
  }
  // identity loss / noise of the NEXT row are put in flight after this row's values have been consumed: a load
  // issued before their last use would share its scoreboard with them
  load_identity_row(L, J, t + 1);
}

// ---- role B: window rows; row t of the ring was written one step earlier
template <class C, class ST>
__device__ __forceinline__ void role_b(const Params& P, const WarpJob& J, int lane, const ST& st, F4* cring,
                                       int t0, int t1, int nit) {
  typedef RoleCfg<C> RC;
  Lane<C> L;
  lane_init(L, P, J, lane);
  // neighbour offsets in the ring (the edge lanes read themselves: their windows are never used)
  const int ol = (lane > 0) ? -1 : 0, orr = (lane < 31) ? 1 : 0;
  load_identity_row(L, J, t0);
  if (role_peel<C>()) {
    role_sync<RC::THREADS>();
#pragma unroll 1
    for (int t = t0; t <= t1; ++t) {
      b_step(L, P, J, lane, st, cring + (t & 1) * RC::NCF4 * 32, t, ol, orr);
      role_sync<RC::THREADS>();
    }
#pragma unroll 1
    for (int i = t1 - t0 + 2; i < nit; ++i) role_sync<RC::THREADS>();
  } else {
#pragma unroll 1
    for (int i = 0; i < nit; ++i) {
      const int t = t0 + i - 1;
      if (i >= 1 && t <= t1) b_step(L, P, J, lane, st, cring + (t & 1) * RC::NCF4 * 32, t, ol, orr);
      role_sync<RC::THREADS>();
    }
  }
  const float ls = warp_sum(L.loss);
  if (lane == 0) atomicAdd(&P.acc[acc_photo(J.s)], (double)ls);
}

// ---- role C, one row: reads its own and its neighbours' coefficients of step t from `q`, stage_c
template <class C, class ST>
__device__ __forceinline__ void c_step(Lane<C>& L, const Params& P, const WarpJob& J, int lane, const ST& st, const F4* q,
                                       int t, int ol, int orr) {
  typedef RoleCfg<C> RC;
  float vc[4 * RC::NCF4], vl[4 * RC::NCF4], vr[4 * RC::NCF4];
#pragma unroll
  for (int k = 0; k < RC::NCF4; ++k) {
    const F4 c = q[k * 32], l = q[k * 32 + ol], r = q[k * 32 + orr];
    vc[4 * k] = c.x; vc[4 * k + 1] = c.y; vc[4 * k + 2] = c.z; vc[4 * k + 3] = c.w;
    vl[4 * k] = l.x; vl[4 * k + 1] = l.y; vl[4 * k + 2] = l.z; vl[4 * k + 3] = l.w;
    vr[4 * k] = r.x; vr[4 * k + 1] = r.y; vr[4 * k + 2] = r.z; vr[4 * k + 3] = r.w;
  }
  Xchg2<C> lf, rt;
#pragma unroll
  for (int n = 0; n < C::NCS; ++n)
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      L.coef[n][k] = vc[n * 9 + k];
      lf.coef[n][k] = vl[n * 9 + k];
      rt.coef[n][k] = vr[n * 9 + k];
    }
  L.tag = __float_as_int(vc[9 * C::NCS]);
  lf.tag = __float_as_int(vl[9 * C::NCS]);
  rt.tag = __float_as_int(vr[9 * C::NCS]);
  wait_target_row<C>(J, st, t - 2);
  stage_c(L, P, J, t, lane, lf, rt, st);
}

template <class C>
__device__ __forceinline__ void c_reduce(const Lane<C>& L, const Params& P, const WarpJob& J, int lane) {
#pragma unroll
  for (int f = 0; f < C::NSRC; ++f) {
    if (!P.pose_grad[f]) continue;
    float dP[12];
    lane_dP(L, P, J, f, dP);
#pragma unroll
    for (int k = 0; k < 12; ++k) {
      const float v = warp_sum(dP[k]);
      if (lane == 0) atomicAdd(&P.acc[acc_dP(P, J.ps, J.b, f, k)], (double)v);
    }
  }
}

// ---- role C: adjoint rows; the coefficients of step t were written one step earlier
template <class C, class ST>
__device__ __forceinline__ void role_c(const Params& P, const WarpJob& J, int lane, const ST& st, const F4* cring,
                                       int t0, int t1, int nit) {
  typedef RoleCfg<C> RC;
  Lane<C> L;
  lane_init(L, P, J, lane);
  const int ol = (lane > 0) ? -1 : 0, orr = (lane < 31) ? 1 : 0;
  stage_next_target_row<C>(J, st, t0, t1, lane);
  if (role_peel<C>()) {
    stage_next_target_row<C>(J, st, t0 + 1, t1, lane);
    role_sync<RC::THREADS>();
    stage_next_target_row<C>(J, st, t0 + 2, t1, lane);
    role_sync<RC::THREADS>();
#pragma unroll 1
    for (int t = t0; t <= t1; ++t) {
      c_step(L, P, J, lane, st, cring + (t & 1) * RC::NCF4 * 32, t, ol, orr);
      stage_next_target_row<C>(J, st, t + 3, t1, lane);
      role_sync<RC::THREADS>();
    }
    c_reduce(L, P, J, lane);
    return;
  }
#pragma unroll 1
  for (int i = 0; i < nit; ++i) {
    const int t = t0 + i - 2;
    if (i >= 2) c_step(L, P, J, lane, st, cring + (t & 1) * RC::NCF4 * 32, t, ol, orr);
    stage_next_target_row<C>(J, st, t0 + i + 1, t1, lane);
    role_sync<RC::THREADS>();
  }
  c_reduce(L, P, J, lane);
}

// ------------------------------------------------------------------ packed-fp32 roles (two sources, per-pixel minimum)
// Roles A and B over the f32x2 stage functions of md2_pack2.cuh (FFMA2 / FADD2 / FMUL2): the scalar FP32
// instructions issue at one per two cycles per scheduler on this part, and role B is the longest of the three
// (494 instructions per row, 312 of them on the fma pipe); packed over the two sources it comes down to the size
// of the other two.  Role C stays scalar (role_c_from_packed).
template <class C, class ST>
__device__ __forceinline__ void role_a2(const Params& P, const WarpJob& J, int lane, const ST& st, int t0, int t1, int nit) {
  Lane2<C> L;
  lane_init2(L, P, J, lane);
  // (--no_ssim: the kernel would land on 136 registers - the 4-CTA trap - or spill under a 128 cap; it keeps the plain form)
  if (role_peel<C>() && C::GRAD && !C::NOSSIM) {
    // projection one row ahead: the depth -> projection -> bilinear-cell chain of row t+1 (no memory access besides the
    // depth of row t+2 put in flight) runs while the gather of row t is in flight; a period then starts with the gather.
    // Two records, two rows per trip: no copy of the record between its computation and its use
    Proj2 Ra, Rb;
    stage_a_proj2<C>(L, Ra, P, J, t0, L.nd[0]);
    prefetch_row2<C, false>(L, J, t0 + 1);
    auto half = [&](int t, Proj2& Rc, Proj2& Rn) {
      stage_a_gather2<C>(L, L.fl, Rc, J, t);
      const float zn = L.nd[0];
      prefetch_row2<C, false>(L, J, t + 2);
      stage_a_proj2<C>(L, Rn, P, J, t + 1, zn);
      L.fl.cz = Rc.cz; L.fl.cu = Rc.cu; L.fl.cv = Rc.cv; L.fl.cwx = Rc.cwx; L.fl.cwy = Rc.cwy; L.fl.cgx = Rc.cgx; L.fl.cgy = Rc.cgy;
      stage_a_finish2<C, ST, true>(L, P, J, t, st);
      role_sync<RoleCfg<C>::THREADS>();
    };
#pragma unroll 1
    for (int t = t0; t <= t1; t += 2) {
      half(t, Ra, Rb);
      if (t + 1 <= t1) half(t + 1, Rb, Ra);
    }
#pragma unroll 1
    for (int p = t1 - t0 + 1; p < nit; ++p) role_sync<RoleCfg<C>::THREADS>();
    return;
  }
  if (role_peel<C>()) {
#pragma unroll 1
    for (int t = t0; t <= t1; ++t) {
      if (!C::GRAD) stage_target_row<C>(J, st, t, lane);
      stage_a_issue2<C, false, 1, true>(L, P, J, t);
      stage_a_finish2<C, ST, true>(L, P, J, t, st);
      role_sync<RoleCfg<C>::THREADS>();
    }
#pragma unroll 1
    for (int p = t1 - t0 + 1; p < nit; ++p) role_sync<RoleCfg<C>::THREADS>();
    return;
  }
#pragma unroll 1
  for (int p = 0; p < nit; ++p) {
    const int t = t0 + p;
    if (t <= t1) {
      if (!C::GRAD) stage_target_row<C>(J, st, t, lane);
      stage_a_issue2<C, false, 1, true>(L, P, J, t);
      stage_a_finish2<C, ST, true>(L, P, J, t, st);
    }
    role_sync<RoleCfg<C>::THREADS>();
  }
}

// Role B's streamed inputs (identity loss and tie-break noise of the two sources) through four running pointers that
// step one image row per loop trip: load_identity_row2 rebuilds the four addresses from the job description every row
// (~38 instructions for 4 loads in the shipped SASS: ptxas rematerialises the base pointers instead of keeping them)
struct IdRows {
  const float* id0; const float* id1; const float* nz0; const float* nz1;
};
template <class C>
__device__ __forceinline__ void id_rows_init(IdRows& R, const Lane2<C>& L, const WarpJob& J, int t) {
  const int yw = t - 1;
  const int pix = (yw < 0 ? 0 : (yw >= J.H ? J.H - 1 : yw)) * J.W + L.xi;
  R.id0 = J.idl + pix; R.id1 = R.id0 + J.plane;
  R.nz0 = J.noise + pix; R.nz1 = R.nz0 + J.plane;
}
// loads the row positioned for step t, then moves to the row of step t + 1 (window row t - 1 clamped to the image)
template <class C>
__device__ __forceinline__ void id_rows_load(Lane2<C>& L, IdRows& R, const WarpJob& J, int t) {
  L.idv[0] = MD2_LDS1(R.id0); L.idv[1] = MD2_LDS1(R.id1);
  L.nzv[0] = MD2_LDS1(R.nz0); L.nzv[1] = MD2_LDS1(R.nz1);
  const int inc = (t >= 1 && t <= J.H - 1) ? J.W : 0;
  R.id0 += inc; R.id1 += inc; R.nz0 += inc; R.nz1 += inc;
}

template <class C, class ST>
__device__ __forceinline__ void b_step2(Lane2<C>& L, const Params& P, const WarpJob& J, int lane, const ST& st, F4* o,
                                        int t, int ol, int orr, IdRows& idr) {
  const int slot = st.slot(t);
  Xchg1P<C> lf, rt;
  wait_target_row<C>(J, st, t);
  const F4* p0 = &st.at(slot, 0, C::STASH4);
  const F4* p1 = &st.at(slot, 1, C::STASH4);
  const F4* p2_ = &st.at(slot, 4, C::STASH4);
  const F4 tc = p0[0], tl = p0[ol], tr = p0[orr];
  const F4 ac = p1[0], al = p1[ol], ar = p1[orr];          // fields 1 / 4 = (r0, g0, r1, g1) / (b0, b1, u0, u1)
  const F4 bc_ = p2_[0], bl = p2_[ol], br = p2_[orr];
  L.tgrg = p2(tc.x, tc.y); L.tgb = tc.z;
  lf.tgrg = p2(tl.x, tl.y); lf.tgb = tl.z;
  rt.tgrg = p2(tr.x, tr.y); rt.tgb = tr.z;
  L.pr[0] = p2(ac.x, ac.y); L.pr[1] = p2(ac.z, ac.w); L.pr[2] = p2(bc_.x, bc_.y);
  lf.pr[0] = p2(al.x, al.y); lf.pr[1] = p2(al.z, al.w); lf.pr[2] = p2(bl.x, bl.y);
  rt.pr[0] = p2(ar.x, ar.y); rt.pr[1] = p2(ar.z, ar.w); rt.pr[2] = p2(br.x, br.y);
  // branch-free form (every lane computes its window, results are selected): 0.3257 vs 0.3295 ms with the divergent one
  stage_b2_straight(L, P, J, t, lane, lf, rt);
  if (C::GRAD) {
    o[0] = make_f4(L.cf[0].x, L.cf[0].y, L.cf[1].x, L.cf[1].y);
    o[32] = make_f4(L.cf[2].x, L.cf[2].y, L.cfb[0], L.cfb[1]);
    o[64] = make_f4(L.cfb[2], __int_as_float(L.tag), 0.f, 0.f);
  }
  if (C::AUTOMASK) id_rows_load(L, idr, J, t + 1);
  else load_identity_row2(L, J, t + 1);
}

template <class C, class ST>
__device__ __forceinline__ void role_b2(const Params& P, const WarpJob& J, int lane, const ST& st, F4* cring,
                                        int t0, int t1, int nit) {
  typedef RoleCfg<C> RC;
  Lane2<C> L;
  lane_init2(L, P, J, lane);
  const int ol = (lane > 0) ? -1 : 0, orr = (lane < 31) ? 1 : 0;
  IdRows idr;
  if (C::AUTOMASK) {
    id_rows_init(idr, L, J, t0);
    id_rows_load(L, idr, J, t0);
  } else load_identity_row2(L, J, t0);
  if (role_peel<C>()) {
    role_sync<RC::THREADS>();                                     // period 0: role A publishes row t0
#pragma unroll 1
    for (int t = t0; t <= t1; ++t) {
      b_step2(L, P, J, lane, st, cring + (t & 1) * RC::NCF4 * 32, t, ol, orr, idr);
      role_sync<RC::THREADS>();
    }
#pragma unroll 1
    for (int i = t1 - t0 + 2; i < nit; ++i) role_sync<RC::THREADS>();
  } else {
#pragma unroll 1
    for (int i = 0; i < nit; ++i) {
      const int t = t0 + i - 1;
      if (i >= 1 && t <= t1) b_step2(L, P, J, lane, st, cring + (t & 1) * RC::NCF4 * 32, t, ol, orr, idr);
      role_sync<RC::THREADS>();
    }
  }
  const float ls = warp_sum(L.loss);
  if (lane == 0) atomicAdd(&P.acc[acc_photo(J.s)], (double)ls);
}

// scalar stage_c fed from the packed coefficient layout of b_step2 (the packed stage C needs a few registers more
// than the 128 that five CTAs per SM leave: 44 bytes of spills; the scalar one fits)
template <class C, class ST>
__device__ __forceinline__ void c_step_from_packed(Lane<C>& L, const Params& P, const WarpJob& J, int lane, const ST& st,
                                                   const F4* q, int t, int ol, int orr) {
  static_assert(C::NCS == 1, "per-pixel minimum");
  auto unpack = [](const F4& a, const F4& b, const F4& c, float* coef, int& tag) {
    coef[0] = a.x; coef[3] = a.y; coef[1] = a.z; coef[4] = a.w; coef[2] = b.x; coef[5] = b.y;
    coef[6] = b.z; coef[7] = b.w; coef[8] = c.x;
    tag = __float_as_int(c.y);
  };
  Xchg2<C> lf, rt;
  unpack(q[0], q[32], q[64], L.coef[0], L.tag);
  unpack(q[ol], q[32 + ol], q[64 + ol], lf.coef[0], lf.tag);
  unpack(q[orr], q[32 + orr], q[64 + orr], rt.coef[0], rt.tag);
  wait_target_row<C>(J, st, t - 2);
  stage_c(L, P, J, t, lane, lf, rt, st);
}

template <class C, class ST>
__device__ __forceinline__ void role_c_from_packed(const Params& P, const WarpJob& J, int lane, const ST& st, const F4* cring,
                                                   int t0, int t1, int nit) {
  typedef RoleCfg<C> RC;
  Lane<C> L;
  lane_init(L, P, J, lane);
  const int ol = (lane > 0) ? -1 : 0, orr = (lane < 31) ? 1 : 0;
  stage_next_target_row<C>(J, st, t0, t1, lane);
  if (role_peel<C>()) {
    // periods 0 and 1: roles A / B fill the rings; this role only stages the next target rows (nit >= 3 always)
    stage_next_target_row<C>(J, st, t0 + 1, t1, lane);
    role_sync<RC::THREADS>();
    stage_next_target_row<C>(J, st, t0 + 2, t1, lane);
    role_sync<RC::THREADS>();
#pragma unroll 1
    for (int t = t0; t <= t1; ++t) {                               // period i = t - t0 + 2
      c_step_from_packed(L, P, J, lane, st, cring + (t & 1) * RC::NCF4 * 32, t, ol, orr);
      stage_next_target_row<C>(J, st, t + 3, t1, lane);
      role_sync<RC::THREADS>();
    }
    c_reduce(L, P, J, lane);
    return;
  }
#pragma unroll 1
  for (int i = 0; i < nit; ++i) {
    const int t = t0 + i - 2;
    if (i >= 2) c_step_from_packed(L, P, J, lane, st, cring + (t & 1) * RC::NCF4 * 32, t, ol, orr);
    stage_next_target_row<C>(J, st, t0 + i + 1, t1, lane);
    role_sync<RC::THREADS>();
  }
  c_reduce(L, P, J, lane);
}

template <class C, bool PACKED>
__global__ void __launch_bounds__(RoleCfg<C>::THREADS) __maxnreg__(RoleCfg<C>::MAXREG) md2_march_roles(Params P) {
  static_assert(!PACKED || (C::NSRC == 2 && !C::AVG), "packed form: two sources, per-pixel minimum");
  typedef RoleCfg<C> RC;
  extern __shared__ float4 smem[];
  const int lane = threadIdx.x & 31;
  // (measured: rotating the warp -> role map from CTA to CTA changes nothing; the hardware does not pin a CTA's
  // warp i to scheduler i % 4 in a way that would pile one role onto one scheduler: per-scheduler issue counts of
  // one launch are within +-10 %)
  const int role = __shfl_sync(kFull, (int)(threadIdx.x >> 5), 0);
  // job order: sample-major (last sample first: the identity pass wrote it most recently, L2), then row segment, scale,
  // band - the scales of one image region read the same target / source rows close together in time; one job per CTA
  const int job = blockIdx.x;
  const int per_seg = P.S * P.nband;
  const int per_b = P.nseg * per_seg;
  const int jb = P.B - 1 - job / per_b;
  const int r = job - (job / per_b) * per_b;
  const int seg = r / per_seg;
  const int r2 = r - seg * per_seg;
  const int js = r2 / P.nband;
  const int jy0 = seg * P.seg_rows;
  WarpJob J = make_job(P, js, jb, (r2 - js * P.nband) * kOwnCols, jy0, min(jy0 + P.seg_rows, P.H));
  // bands whose 32 lanes all lie inside the image: the target row is staged by TMA (others read reflected columns)
  // (1-2 sources: measured on one box 0.389 vs 0.419 ms at 640x192, 1.017 vs 1.071 ms at 1024x320; the 3-source
  // kernels, at their register limit, lose: 0.533 vs 0.499 ms, and keep the per-lane loads)
  if (C::NSRC <= 2) J.staged = (J.x0 - 2 >= 0) && (J.x0 + 30 <= J.W);

  StashT<RC::RING> st;
  st.base = smem + lane;
  st.bring = nullptr;
  st.stride = 32;
  st.tbar = reinterpret_cast<unsigned long long*>(smem + RC::STASH_F4 + RC::COEF_F4);
  F4* cring = smem + RC::STASH_F4 + lane;
  const int t0 = J.y0 - 2, t1 = J.y1 + 1;
  st.t0 = t0;
  const int nit = (t1 - t0 + 1) + (C::GRAD ? 2 : 1);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < RC::RING; ++i) mbar_init(st.tbar + i, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if constexpr (PACKED) {
    typedef PairedOf<C> CP;
    if (role < RC::NA) role_a2<CP>(P, J, lane, st, t0, t1, nit);
    else if (role == RC::NA) role_b2<CP>(P, J, lane, st, cring, t0, t1, nit);
    else if (C::GRAD) role_c_from_packed<CP>(P, J, lane, st, cring, t0, t1, nit);
  } else {
    if (role < RC::NA) role_a<C>(P, J, lane, st, t0, t1, nit);
    else if (role == RC::NA) role_b<C>(P, J, lane, st, cring, t0, t1, nit);
    else if (C::GRAD) role_c<C>(P, J, lane, st, cring, t0, t1, nit);
  }
}

}  // namespace md2
