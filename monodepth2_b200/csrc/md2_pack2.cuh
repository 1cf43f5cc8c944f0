// md2_pack2.cuh - packed-fp32 (FFMA2 / FADD2 / FMUL2, sm_100a) form of the marching kernel's per-lane
// arithmetic for TWO sources without --avg_reprojection (the headline configuration).
//
// Same algorithm, same order of operations and same stash layout as the scalar stage functions of
// md2_core.cuh (which stay the single source for 1 / 3 sources, --avg_reprojection and the host
// emulator); what changes is the register layout:
//   * stage A (projection):   every per-source scalar is a float2 over the two sources (f0, f1)
//   * stage A (interpolation): per source, channels (r,g) are a float2 straight out of the RGBx
//                              LDG.128 (x,y are an aligned register pair), b is scalar
//   * stage B (window sums, SSIM): 6 (source, channel) values = 3 slots
//                              slot0 = (r,g) of source 0, slot1 = (r,g) of source 1, slot2 = (b of 0, b of 1);
//                              the target partner of slots 0/1 is the (r,g) pair of the target texel, of
//                              slot 2 the scalar b (a scalar operand of an f32x2 instruction is broadcast
//                              by the hardware: `FFMA2 R, R.F32, R.F32x2, imm`, no register moves)
//   * stage C (adjoint):      the winner's SSIM-adjoint coefficients are float2 over (r,g) + scalar b;
//                              box sums per source the same; the b sums, the pose sums and the projection
//                              rows are float2 over the two sources
// ~37 % fewer FP32 issue slots than the scalar form (static loop 1245 -> 1067 instructions).  Measured on
// B200 (profiles/r01_optimization_log.md): the forward-only kernel (154 registers, 12 warps per SM) gets
// 23 % faster (0.272 -> 0.209 ms), the forward+adjoint kernel sits at the 255-register cap either way and
// is latency-bound at 8 warps per SM: 0.443 ms packed vs 0.427 ms scalar.  The role-specialised kernel
// (md2_roles.cuh) runs its roles A and B in this form for two sources without --avg_reprojection (except
// --disable_automasking with gradients), and so does the identity pass; MD2_PACK2=off in the environment
// forces the scalar form (A/B tests).
// Device-only (the emulator keeps the scalar form; tests/test_gpu_parity.py ties the two together).
#pragma once

#include "md2_core.cuh"

#if defined(__CUDACC__)

namespace md2 {

typedef float2 P2;
__device__ __forceinline__ P2 p2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ P2 bc(float a) { return make_float2(a, a); }              // broadcast operand
__device__ __forceinline__ P2 neg2(P2 a) { return make_float2(-a.x, -a.y); }         // folds into the operand modifier
__device__ __forceinline__ P2 fma2(P2 a, P2 b, P2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ P2 add2(P2 a, P2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ P2 sub2(P2 a, P2 b) { return __fadd2_rn(a, neg2(b)); }
__device__ __forceinline__ P2 mul2(P2 a, P2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ P2 sel2(bool c, P2 a, P2 b) { return c ? a : b; }
__device__ __forceinline__ float rcp_fast(float a) {      // MUFU.RCP (nvcc's host pass only parses this)
#if defined(__CUDA_ARCH__)
  return rcp_approx(a);
#else
  return 1.0f / a;
#endif
}

// SSIM of two windows at once (see ssim_window in md2_core.cuh for the algebra).
// coef (optional) receives -0.5*live*(alpha, beta, gamma) as three pairs.
__device__ __forceinline__ P2 ssim_window2(P2 sx, P2 sxx, P2 sxy, P2 sy, P2 syy, P2* coef) {
  const P2 c1 = bc(81.0f * kSsimC1), c2 = bc(81.0f * kSsimC2);
  const P2 pxy = mul2(sx, sy);
  const P2 pp = fma2(sx, sx, mul2(sy, sy));
  const P2 n1 = fma2(bc(2.0f), pxy, c1);
  const P2 n2 = fma2(bc(2.0f), fma2(bc(9.0f), sxy, neg2(pxy)), c2);
  const P2 d1 = add2(pp, c1);
  const P2 d2 = add2(fma2(bc(9.0f), add2(sxx, syy), neg2(pp)), c2);
  const P2 N = mul2(n1, n2), D = mul2(d1, d2);
  const P2 invD = p2(MD2_RCP_SSIM(D.x), MD2_RCP_SSIM(D.y));
  const P2 Q = mul2(N, invD);
  const P2 raw = fma2(bc(-0.5f), Q, bc(0.5f));
  const P2 S = p2(fminf(fmaxf(raw.x, 0.0f), 1.0f), fminf(fmaxf(raw.y, 0.0f), 1.0f));
  if (coef) {
    const P2 k = p2(((raw.x >= 0.0f) && (raw.x <= 1.0f)) ? -0.5f : 0.0f,
                    ((raw.y >= 0.0f) && (raw.y <= 1.0f)) ? -0.5f : 0.0f);
    const P2 QD = mul2(Q, invD);                       // N / D^2
    const P2 a1 = mul2(mul2(sy, sub2(n2, n1)), invD);
    const P2 a2 = mul2(mul2(sx, sub2(d2, d1)), QD);
    const P2 alpha = mul2(bc(2.0f), sub2(a1, a2));
    const P2 beta = mul2(mul2(bc(-18.0f), d1), QD);
    const P2 gamma = mul2(mul2(bc(18.0f), n1), invD);
    coef[0] = mul2(k, alpha);
    coef[1] = mul2(k, beta);
    coef[2] = mul2(k, gamma);
  }
  return S;
}

// ------------------------------------------------------------------ lane state (two sources)
struct Flight2 {                   // see Flight (md2_core.cuh)
  F4 tap[2][4];
  float cz;
  P2 cu, cv, cwx, cwy, cgx, cgy;   // over the two sources
  F4 ctg;
};
// the part of a Flight2 that does not depend on the gathered texels (role A computes it one row ahead, in the shadow of
// the previous row's gather: stage_a_proj2 / stage_a_gather2)
struct Proj2 {
  float cz;
  P2 cu, cv, cwx, cwy, cgx, cgy;
  int toff[2], dx1[2], dy1[2];     // per source: float offset of the north-west texel, steps to the east / south tap
};

template <class C>
struct Lane2 {
  int x, xi;
  bool colok;
  P2 qa[3], qb[3], p4[3];          // over the two sources: M[i][0]*xi + M[i][2] | M[i][1] | (K T)[i][3]
  int ux0, ux1;
  float ul0, ul1;
  F4 ntg;
  float nd[4];
  Flight2 fl;                      // gather of the current row, in flight between issue and finish
  float idv[2], nzv[2];
  // forward rolling state: [slot][x, xx, xy]; target: (r,g) pair and scalar b, [y, yy]
  P2 H1[3][3], H2[3][3];
  P2 HYrg1[2], HYrg2[2];
  float HYb1[2], HYb2[2];
  P2 pr1[3], tgrg1;
  float tgb1;
  P2 pr[3], tgrg;                  // exports of the current step (slots)
  float tgb;
  P2 cf[3];                        // winner's (alpha, beta, gamma) over (r,g)
  float cfb[3];                    // ... of channel b
  int tag;
  // backward rolling state
  P2 B1rg[2][3], B2rg[2][3];       // [source][alpha,beta,gamma] over (r,g)
  P2 B1b[3], B2b[3];               // channel b, over the two sources
  int tag1;
  float loss;
  P2 S1[3], S2[3], S3[3];          // pose sums over the two sources
};

template <class C>
struct Xchg1P {
  P2 pr[3];
  P2 tgrg;
  float tgb;
};

template <class C, bool WITH_TG = true>
__device__ __forceinline__ void prefetch_row2(Lane2<C>& L, const WarpJob& J, int t) {
  const int tr = reflect_clamp(t, J.H);
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
    L.nd[0] = MD2_LD(r0 + L.ux0); L.nd[1] = MD2_LD(r0 + L.ux1);
    L.nd[2] = MD2_LD(r1 + L.ux0); L.nd[3] = MD2_LD(r1 + L.ux1);
  }
}

template <class C>
__device__ __forceinline__ void lane_init2(Lane2<C>& L, const Params& P, const WarpJob& J, int lane) {
  L.x = J.x0 - 2 + lane;
  L.colok = (L.x >= 0) && (L.x < P.W);
  L.xi = reflect_clamp(L.x, P.W);
  const float xf = (float)L.xi;
  const float* m0 = J.proj;
  const float* m1 = m0 + 12;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    L.qa[i] = p2(fmaf(MD2_LD(m0 + i * 3 + 0), xf, MD2_LD(m0 + i * 3 + 2)),
                 fmaf(MD2_LD(m1 + i * 3 + 0), xf, MD2_LD(m1 + i * 3 + 2)));
    L.qb[i] = p2(MD2_LD(m0 + i * 3 + 1), MD2_LD(m1 + i * 3 + 1));
    L.p4[i] = p2(MD2_LD(m0 + 9 + i), MD2_LD(m1 + 9 + i));
  }
  L.idv[0] = L.idv[1] = L.nzv[0] = L.nzv[1] = 0.f;
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
  const P2 z2 = bc(0.f);
#pragma unroll
  for (int s = 0; s < 3; ++s) {
#pragma unroll
    for (int k = 0; k < 3; ++k) { L.H1[s][k] = z2; L.H2[s][k] = z2; }
    L.pr1[s] = z2; L.pr[s] = z2;
    L.S1[s] = z2; L.S2[s] = z2; L.S3[s] = z2;
    L.cf[s] = z2; L.cfb[s] = 0.f;
    L.B1b[s] = z2; L.B2b[s] = z2;
#pragma unroll
    for (int f = 0; f < 2; ++f) { L.B1rg[f][s] = z2; L.B2rg[f][s] = z2; }
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) { L.HYrg1[k] = z2; L.HYrg2[k] = z2; L.HYb1[k] = 0.f; L.HYb2[k] = 0.f; }
  L.tgrg1 = z2; L.tgrg = z2; L.tgb1 = 0.f; L.tgb = 0.f;
  L.tag = -1; L.tag1 = -1;
  L.loss = 0.f;
  prefetch_row2(L, J, J.y0 - 2);
}

// ------------------------------------------------------------------ stage A (see stage_a_issue / stage_a_finish)
template <class C>
__device__ __forceinline__ void load_identity_row2(Lane2<C>& L, const WarpJob& J, int t) {
  if (C::AUTOMASK) {
    const int yw = t - 1;
    const int pix = (yw < 0 ? 0 : (yw >= J.H ? J.H - 1 : yw)) * J.W + L.xi;
    L.idv[0] = MD2_LDS1(J.idl + pix);
    L.idv[1] = MD2_LDS1(J.idl + J.plane + pix);
    L.nzv[0] = MD2_LDS1(J.noise + pix);
    L.nzv[1] = MD2_LDS1(J.noise + J.plane + pix);
  } else if (J.pm) {       // --predictive_mask: see load_identity_row
    const int yw = t - 1;
    const int pix = (yw < 0 ? 0 : (yw >= J.H ? J.H - 1 : yw)) * J.W + L.xi;
    L.nzv[0] = MD2_LDS1(J.pm + pix);
    L.nzv[1] = MD2_LDS1(J.pm + J.plane + pix);
  }
}

template <class C, bool WITH_ID = true, int ROW_STEP = 1, bool TG_DIRECT = false>
__device__ __forceinline__ void stage_a_issue2(Lane2<C>& L, Flight2& F, const Params& P, const WarpJob& J, int t) {
  const int tr = reflect_clamp(t, J.H);
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
  if (ROW_STEP > 0) prefetch_row2<C, !TG_DIRECT>(L, J, t + ROW_STEP);
  if (WITH_ID) load_identity_row2(L, J, t);
  const float z = C::ZUP ? (J.s == 0 ? depth_of_disp(P, zpre) : zpre) : depth_of_disp(P, D);
  F.cz = z;
  const float yf = (float)tr;
  const P2 q0 = fma2(L.qb[0], bc(yf), L.qa[0]);
  const P2 q1 = fma2(L.qb[1], bc(yf), L.qa[1]);
  const P2 q2 = fma2(L.qb[2], bc(yf), L.qa[2]);
  const P2 c0 = fma2(bc(z), q0, L.p4[0]);
  const P2 c1 = fma2(bc(z), q1, L.p4[1]);
  const P2 c2 = fma2(bc(z), q2, L.p4[2]);
  const P2 den = add2(c2, bc(P.eps));
  const P2 r0 = p2(rcp_fast(den.x), rcp_fast(den.y));
  const P2 inv = fma2(r0, fma2(neg2(den), r0, bc(1.0f)), r0);      // Newton step of rcp_nr
  const P2 u = mul2(c0, inv);
  const P2 v = mul2(c1, inv);
  const P2 ix = fma2(u, bc(P.sx), bc(P.ox));
  const P2 iy = fma2(v, bc(P.sy), bc(P.oy));
  const P2 ixc = p2(fminf(fmaxf(ix.x, 0.0f), P.wmax), fminf(fmaxf(ix.y, 0.0f), P.wmax));
  const P2 iyc = p2(fminf(fmaxf(iy.x, 0.0f), P.hmax), fminf(fmaxf(iy.y, 0.0f), P.hmax));
  const P2 fx0 = p2(floorf(ixc.x), floorf(ixc.y));
  const P2 fy0 = p2(floorf(iyc.x), floorf(iyc.y));
  const P2 gx = mul2(bc(P.sx), inv), gy = mul2(bc(P.sy), inv);
  F.cu = u; F.cv = v;
  F.cwx = sub2(ixc, fx0); F.cwy = sub2(iyc, fy0);
  F.cgx = p2(((ix.x > 0.0f) && (ix.x < P.wmax)) ? gx.x : 0.0f, ((ix.y > 0.0f) && (ix.y < P.wmax)) ? gx.y : 0.0f);
  F.cgy = p2(((iy.x > 0.0f) && (iy.x < P.hmax)) ? gy.x : 0.0f, ((iy.y > 0.0f) && (iy.y < P.hmax)) ? gy.y : 0.0f);
#pragma unroll
  for (int f = 0; f < 2; ++f) {
    const int x0 = (int)(f ? fx0.y : fx0.x), y0 = (int)(f ? fy0.y : fy0.x);
    const int dx1 = (x0 + 1 < J.W) ? 4 : 0;
    const int dy1 = (y0 + 1 < J.H) ? J.W * 4 : 0;
    const float* t00 = J.src4[f] + 4 * (y0 * J.W + x0);
    F.tap[f][0] = MD2_LD4(t00);
    F.tap[f][1] = MD2_LD4(t00 + dx1);
    F.tap[f][2] = MD2_LD4(t00 + dy1);
    F.tap[f][3] = MD2_LD4(t00 + dy1 + dx1);
  }
}

template <class C, bool WITH_ID = true, int ROW_STEP = 1, bool TG_DIRECT = false>
__device__ __forceinline__ void stage_a_issue2(Lane2<C>& L, const Params& P, const WarpJob& J, int t) {
  stage_a_issue2<C, WITH_ID, ROW_STEP, TG_DIRECT>(L, L.fl, P, J, t);
}

// stage_a_issue2 in two halves (Cfg::ZUP kernels): everything up to the tap addresses of row t ...
template <class C>
__device__ __forceinline__ void stage_a_proj2(Lane2<C>& L, Proj2& R, const Params& P, const WarpJob& J, int t, float zrow) {
  const int tr = reflect_clamp(t, J.H);
  const float z = (J.s == 0) ? depth_of_disp(P, zrow) : zrow;
  R.cz = z;
  const float yf = (float)tr;
  const P2 q0 = fma2(L.qb[0], bc(yf), L.qa[0]);
  const P2 q1 = fma2(L.qb[1], bc(yf), L.qa[1]);
  const P2 q2 = fma2(L.qb[2], bc(yf), L.qa[2]);
  const P2 c0 = fma2(bc(z), q0, L.p4[0]);
  const P2 c1 = fma2(bc(z), q1, L.p4[1]);
  const P2 c2 = fma2(bc(z), q2, L.p4[2]);
  const P2 den = add2(c2, bc(P.eps));
  const P2 r0 = p2(rcp_fast(den.x), rcp_fast(den.y));
  const P2 inv = fma2(r0, fma2(neg2(den), r0, bc(1.0f)), r0);      // Newton step of rcp_nr
  const P2 u = mul2(c0, inv);
  const P2 v = mul2(c1, inv);
  const P2 ix = fma2(u, bc(P.sx), bc(P.ox));
  const P2 iy = fma2(v, bc(P.sy), bc(P.oy));
  const P2 ixc = p2(fminf(fmaxf(ix.x, 0.0f), P.wmax), fminf(fmaxf(ix.y, 0.0f), P.wmax));
  const P2 iyc = p2(fminf(fmaxf(iy.x, 0.0f), P.hmax), fminf(fmaxf(iy.y, 0.0f), P.hmax));
  const P2 fx0 = p2(floorf(ixc.x), floorf(ixc.y));
  const P2 fy0 = p2(floorf(iyc.x), floorf(iyc.y));
  const P2 gx = mul2(bc(P.sx), inv), gy = mul2(bc(P.sy), inv);
  R.cu = u; R.cv = v;
  R.cwx = sub2(ixc, fx0); R.cwy = sub2(iyc, fy0);
  R.cgx = p2(((ix.x > 0.0f) && (ix.x < P.wmax)) ? gx.x : 0.0f, ((ix.y > 0.0f) && (ix.y < P.wmax)) ? gx.y : 0.0f);
  R.cgy = p2(((iy.x > 0.0f) && (iy.x < P.hmax)) ? gy.x : 0.0f, ((iy.y > 0.0f) && (iy.y < P.hmax)) ? gy.y : 0.0f);
#pragma unroll
  for (int f = 0; f < 2; ++f) {
    const int x0 = (int)(f ? fx0.y : fx0.x), y0 = (int)(f ? fy0.y : fy0.x);
    R.toff[f] = 4 * (y0 * J.W + x0);
    R.dx1[f] = (x0 + 1 < J.W) ? 4 : 0;
    R.dy1[f] = (y0 + 1 < J.H) ? J.W * 4 : 0;
  }
}
// ... and the gather itself (plus the target texel of bands that are not staged by TMA); the caller moves the rest of
// the record into F after its next stage_a_proj2
template <class C>
__device__ __forceinline__ void stage_a_gather2(const Lane2<C>& L, Flight2& F, const Proj2& R, const WarpJob& J, int t) {
  if (J.staged) F.ctg = make_f4(0.f, 0.f, 0.f, 0.f);
  else F.ctg = MD2_LDS4(J.tgt4 + 4 * (reflect_clamp(t, J.H) * J.W + L.xi));
#pragma unroll
  for (int f = 0; f < 2; ++f) {
    const int dx1 = R.dx1[f], dy1 = R.dy1[f];
    const float* t00 = J.src4[f] + R.toff[f];
    F.tap[f][0] = MD2_LD4(t00);
    F.tap[f][1] = MD2_LD4(t00 + dx1);
    F.tap[f][2] = MD2_LD4(t00 + dy1);
    F.tap[f][3] = MD2_LD4(t00 + dy1 + dx1);
  }
}

template <class C, class ST, bool PUBLISH = C::GRAD>
__device__ __forceinline__ void stage_a_finish2(Lane2<C>& L, const Flight2& F, const Params& P, const WarpJob& J, int t, const ST& st) {
  const int slot = st.slot(t);
  const F4 tg4 = F.ctg;
  const float z = F.cz;
  const bool own = (t >= J.y0) && (t < J.y1) && (L.x >= J.x0) && (L.x < J.x0 + kOwnCols) && L.colok;
  L.tgrg = p2(tg4.x, tg4.y);
  L.tgb = tg4.z;
  if (J.depth && own) J.depth[t * J.W + L.xi] = z;
  if (PUBLISH && !J.staged) st.at(slot, 0, C::STASH4) = make_f4(tg4.x, tg4.y, tg4.z, 0.f);   // see stage_a_finish
  float prb[2];
#pragma unroll
  for (int f = 0; f < 2; ++f) {
    const F4 nw = F.tap[f][0], ne = F.tap[f][1], sw = F.tap[f][2], se = F.tap[f][3];
    const float wx = f ? F.cwx.y : F.cwx.x, wy = f ? F.cwy.y : F.cwy.x;
    const float gxs = f ? F.cgx.y : F.cgx.x, gys = f ? F.cgy.y : F.cgy.x;
    // channels (r,g) as a pair
    const P2 nw2 = p2(nw.x, nw.y), ne2 = p2(ne.x, ne.y), sw2 = p2(sw.x, sw.y), se2 = p2(se.x, se.y);
    const P2 dn2 = sub2(ne2, nw2), ds2 = sub2(se2, sw2);
    const P2 top2 = fma2(bc(wx), dn2, nw2), bot2 = fma2(bc(wx), ds2, sw2);
    const P2 dv2 = sub2(bot2, top2);
    const P2 pr2 = fma2(bc(wy), dv2, top2);
    const P2 dxp2 = mul2(fma2(bc(wy), sub2(ds2, dn2), dn2), bc(gxs));
    const P2 dyp2 = mul2(dv2, bc(gys));
    // channel b
    const float dn = ne.z - nw.z, ds = se.z - sw.z;
    const float top = fmaf(wx, dn, nw.z), bot = fmaf(wx, ds, sw.z);
    const float dv = bot - top;
    const float pb = fmaf(wy, dv, top);
    const float dxb = fmaf(wy, ds - dn, dn) * gxs;
    const float dyb = dv * gys;
    if (J.warped[f] && own) {
      float* w = J.warped[f] + t * J.W + L.xi;
      w[0] = pr2.x; w[J.plane] = pr2.y; w[2 * J.plane] = pb;
    }
    L.pr[f] = pr2;
    prb[f] = pb;
    if (PUBLISH && !C::PAIRED) st.at(slot, 1 + 3 * f, C::STASH4) = make_f4(pr2.x, pr2.y, pb, f ? F.cu.y : F.cu.x);
    if (C::GRAD) {
      st.at(slot, 2 + 3 * f, C::STASH4) = make_f4(dxp2.x, dxp2.y, dxb, f ? F.cv.y : F.cv.x);
      st.at(slot, 3 + 3 * f, C::STASH4) = make_f4(dyp2.x, dyp2.y, dyb, f == 0 ? z : 0.f);
    }
  }
  L.pr[2] = p2(prb[0], prb[1]);
  if (PUBLISH && C::PAIRED) {
    st.at(slot, 1, C::STASH4) = make_f4(L.pr[0].x, L.pr[0].y, L.pr[1].x, L.pr[1].y);
    st.at(slot, 4, C::STASH4) = make_f4(prb[0], prb[1], F.cu.x, F.cu.y);
  }
}

template <class C, class ST, bool PUBLISH = C::GRAD>
__device__ __forceinline__ void stage_a_finish2(Lane2<C>& L, const Params& P, const WarpJob& J, int t, const ST& st) {
  stage_a_finish2<C, ST, PUBLISH>(L, L.fl, P, J, t, st);
}

// ------------------------------------------------------------------ stage B (see stage_b_straight)
// Branch-free: every lane computes the window, results are selected.
template <class C>
__device__ __forceinline__ void stage_b2_straight(Lane2<C>& L, const Params& P, const WarpJob& J, int t, int lane,
                                         const Xchg1P<C>& lf, const Xchg1P<C>& rt) {
  const int yw = t - 1;
  P2 H0[3][3], HYrg0[2];
  float HYb0[2];
  HYrg0[0] = add2(add2(lf.tgrg, L.tgrg), rt.tgrg);
  HYrg0[1] = fma2(rt.tgrg, rt.tgrg, fma2(L.tgrg, L.tgrg, mul2(lf.tgrg, lf.tgrg)));
  HYb0[0] = lf.tgb + L.tgb + rt.tgb;
  HYb0[1] = fmaf(rt.tgb, rt.tgb, fmaf(L.tgb, L.tgb, lf.tgb * lf.tgb));
#pragma unroll
  for (int s = 0; s < 3; ++s) {
    const P2 yl = (s < 2) ? lf.tgrg : bc(lf.tgb), yc = (s < 2) ? L.tgrg : bc(L.tgb), yr = (s < 2) ? rt.tgrg : bc(rt.tgb);
    const P2 xl = lf.pr[s], xc = L.pr[s], xr = rt.pr[s];
    H0[s][0] = add2(add2(xl, xc), xr);
    H0[s][1] = fma2(xr, xr, fma2(xc, xc, mul2(xl, xl)));
    H0[s][2] = fma2(xr, yr, fma2(xc, yc, mul2(xl, yl)));
  }
  const bool win_ok = L.colok && (yw >= 0) && (yw < P.H) && (lane >= 1) && (lane <= kLanes - 2) &&
                      (yw >= J.y0 - (C::GRAD ? 1 : 0)) && (yw < J.y1 + (C::GRAD ? 1 : 0));
  const bool own_win = win_ok && (lane >= 2) && (lane < 2 + kOwnCols) && (yw >= J.y0) && (yw < J.y1);
  int tag = -1;
#pragma unroll
  for (int i = 0; i < 3; ++i) { L.cf[i] = bc(0.f); L.cfb[i] = 0.f; }
  {
    P2 V[3][3], VYrg[2];
    float VYb[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) { VYrg[k] = add2(L.HYrg2[k], HYrg0[k]); VYb[k] = L.HYb2[k] + HYb0[k]; }
#pragma unroll
    for (int s = 0; s < 3; ++s)
#pragma unroll
      for (int k = 0; k < 3; ++k) V[s][k] = add2(L.H2[s][k], H0[s][k]);
    P2 S[3];
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      S[s] = bc(0.f);
      if (!C::NOSSIM)
        S[s] = ssim_window2(V[s][0], V[s][1], V[s][2], (s < 2) ? VYrg[0] : bc(VYb[0]), (s < 2) ? VYrg[1] : bc(VYb[1]), nullptr);
    }
    const P2 e0 = sub2(L.tgrg1, L.pr1[0]), e1 = sub2(L.tgrg1, L.pr1[1]), e2 = sub2(bc(L.tgb1), L.pr1[2]);
    float rl[2];
    {
      const float ss0 = ((0.f + S[0].x) + S[0].y) + S[2].x, ss1 = ((0.f + S[1].x) + S[1].y) + S[2].y;
      const float l10 = ((0.f + fabsf(e0.x)) + fabsf(e0.y)) + fabsf(e2.x);
      const float l11 = ((0.f + fabsf(e1.x)) + fabsf(e1.y)) + fabsf(e2.y);
      rl[0] = C::NOSSIM ? l10 * (1.0f / 3.0f) : fmaf(0.85f / 3.0f, ss0, (0.15f / 3.0f) * l10);
      rl[1] = C::NOSSIM ? l11 * (1.0f / 3.0f) : fmaf(0.85f / 3.0f, ss1, (0.15f / 3.0f) * l11);
    }
    float best = INFINITY;
    if (C::AUTOMASK) {
#pragma unroll
      for (int f = 0; f < 2; ++f) {
        const float cand = MD2_FADD(L.idv[f], MD2_FMUL(L.nzv[f], 0.00001f));
        if (cand < best) best = cand;
      }
    }
    const bool pm = !C::AUTOMASK && J.pm;             // --predictive_mask (see pmask_apply in md2_core.cuh)
#pragma unroll
    for (int f = 0; f < 2; ++f) {
      const float cand = pm ? rl[f] * L.nzv[f] : rl[f];
      if (cand < best) { best = cand; tag = f; }
    }
    L.loss += own_win ? best : 0.0f;
    if (own_win) {
      if (C::AUTOMASK && J.idsel) J.idsel[yw * J.W + L.xi] = (tag >= 0) ? 1.0f : 0.0f;
      if (pm && C::GRAD && J.gpm) {
#pragma unroll
        for (int f = 0; f < 2; ++f) J.gpm[f * J.plane + yw * J.W + L.xi] = (tag == f) ? rl[f] * P.gscale : 0.0f;
      }
    }
    if (!win_ok) tag = -1;
    if (C::GRAD && !C::NOSSIM) {
      // the winner's window sums: (r,g) pair from slot `tag`, b from that half of slot 2
      const bool w1 = (tag == 1);
      P2 Wrg[3];
      float Wb[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) { Wrg[k] = sel2(w1, V[1][k], V[0][k]); Wb[k] = w1 ? V[2][k].y : V[2][k].x; }
      ssim_window2(Wrg[0], Wrg[1], Wrg[2], VYrg[0], VYrg[1], L.cf);
      ssim_window(Wb[0], Wb[1], Wb[2], VYb[0], VYb[1], L.cfb);
      if (pm) {
        const float m = w1 ? L.nzv[1] : L.nzv[0];
#pragma unroll
        for (int k = 0; k < 3; ++k) { L.cf[k] = mul2(L.cf[k], bc(m)); L.cfb[k] *= m; }
      }
      // selects, not products: lanes without a window (or whose identity candidate won) may hold non-finite sums
      const bool live = tag >= 0;
#pragma unroll
      for (int k = 0; k < 3; ++k) { L.cf[k] = sel2(live, L.cf[k], bc(0.f)); L.cfb[k] = live ? L.cfb[k] : 0.0f; }
    }
  }
  L.tag = tag;
  // roll the forward state
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    L.HYrg2[k] = add2(L.HYrg1[k], HYrg0[k]); L.HYrg1[k] = HYrg0[k];
    L.HYb2[k] = L.HYb1[k] + HYb0[k]; L.HYb1[k] = HYb0[k];
  }
  L.tgrg1 = L.tgrg; L.tgb1 = L.tgb;
#pragma unroll
  for (int s = 0; s < 3; ++s) {
#pragma unroll
    for (int k = 0; k < 3; ++k) { L.H2[s][k] = add2(L.H1[s][k], H0[s][k]); L.H1[s][k] = H0[s][k]; }
    L.pr1[s] = L.pr[s];
  }
}

// lane's share of dP for source f (see lane_dP)
template <class C>
__device__ __forceinline__ void lane_dP2(const Lane2<C>& L, const Params& P, const WarpJob& J, int f, float* dP) {
  const float* ik = P.invK + (size_t)J.b * 16;
  const float xf = (float)L.xi;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float ak = fmaf(MD2_LD(ik + k * 4 + 0), xf, MD2_LD(ik + k * 4 + 2));
    const float bk = MD2_LD(ik + k * 4 + 1);
#pragma unroll
    for (int i = 0; i < 3; ++i) dP[i * 4 + k] = fmaf(ak, f ? L.S1[i].y : L.S1[i].x, bk * (f ? L.S2[i].y : L.S2[i].x));
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) dP[i * 4 + 3] = f ? L.S3[i].y : L.S3[i].x;
}

// ------------------------------------------------------------------ identity pass, two sources (see id_stage_a / id_stage_b)
struct IdLane2 {
  int x, xi;
  bool colok;
  P2 H1[3][3], H2[3][3];
  P2 HYrg1[2], HYrg2[2];
  float HYb1[2], HYb2[2];
  P2 pr1[3], tgrg1;
  float tgb1;
  P2 pr[3], tgrg;
  float tgb;
  float npr[2][3], ntg[3];        // row t+1, in flight
  float n2pr[2][3], n2tg[3];      // row t+2, in flight (the pass is bound by bytes in flight, not by issue)
};
struct IdXchg2 {
  P2 pr[3];
  P2 tgrg;
  float tgb;
};

__device__ __forceinline__ void id_init2(IdLane2& L, const Params& P, int x0, int lane) {
  L.x = x0 - 1 + lane;
  L.colok = (L.x >= 0) && (L.x < P.W);
  L.xi = reflect_clamp(L.x, P.W);
  const P2 z2 = bc(0.f);
#pragma unroll
  for (int s = 0; s < 3; ++s) {
#pragma unroll
    for (int k = 0; k < 3; ++k) { L.H1[s][k] = z2; L.H2[s][k] = z2; }
    L.pr1[s] = z2; L.pr[s] = z2;
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) { L.HYrg1[k] = z2; L.HYrg2[k] = z2; L.HYb1[k] = 0.f; L.HYb2[k] = 0.f; }
  L.tgrg1 = z2; L.tgrg = z2; L.tgb1 = 0.f; L.tgb = 0.f;
}

// issue the planar loads of row t into the far prefetch slot (consumed two steps later)
__device__ __forceinline__ void id_prefetch2(IdLane2& L, const Params& P, int b, int t) {
  const int tr = reflect_clamp(t, P.H);
  const int plane = P.H * P.W;
  const int pix = tr * P.W + L.xi;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    L.n2tg[c] = load_px(P.tgt, P.tgt8, P.u8_hwc, b, c, plane, pix);
    L.n2pr[0][c] = load_px(P.src[0], P.src8[0], P.u8_hwc, b, c, plane, pix);
    L.n2pr[1][c] = load_px(P.src[1], P.src8[1], P.u8_hwc, b, c, plane, pix);
  }
}
__device__ __forceinline__ void id_shift2(IdLane2& L) {
#pragma unroll
  for (int c = 0; c < 3; ++c) { L.ntg[c] = L.n2tg[c]; L.npr[0][c] = L.n2pr[0][c]; L.npr[1][c] = L.n2pr[1][c]; }
}

__device__ __forceinline__ void id_stage_a2(IdLane2& L, const Params& P, int b, int t, int lane, int y0, int y1) {
  const int tr = reflect_clamp(t, P.H);
  const int plane = P.H * P.W;
  const bool own = L.colok && t >= y0 && t < y1 && lane >= 1 && lane <= kIdCols;
  const int o4 = 4 * (b * plane + tr * P.W + L.xi);
  const float tg[3] = {L.ntg[0], L.ntg[1], L.ntg[2]};
  const float p0[3] = {L.npr[0][0], L.npr[0][1], L.npr[0][2]}, p1[3] = {L.npr[1][0], L.npr[1][1], L.npr[1][2]};
  L.tgrg = p2(tg[0], tg[1]); L.tgb = tg[2];
  L.pr[0] = p2(p0[0], p0[1]); L.pr[1] = p2(p1[0], p1[1]); L.pr[2] = p2(p0[2], p1[2]);
  id_shift2(L);
  id_prefetch2(L, P, b, t + 2);
  if (own) {
    *reinterpret_cast<F4*>(P.tgt4 + o4) = make_f4(tg[0], tg[1], tg[2], 0.f);
    *reinterpret_cast<F4*>(P.src4[0] + o4) = make_f4(p0[0], p0[1], p0[2], 0.f);
    *reinterpret_cast<F4*>(P.src4[1] + o4) = make_f4(p1[0], p1[1], p1[2], 0.f);
  }
}

template <bool NOSSIM>
__device__ __forceinline__ void id_stage_b2(IdLane2& L, const Params& P, int b, int t, int lane, int y0, int y1,
                                            const IdXchg2& lf, const IdXchg2& rt, int lane_lo = 1, int lane_hi = kIdCols) {
  const int yw = t - 1;
  P2 H0[3][3], HYrg0[2];
  float HYb0[2];
  HYrg0[0] = add2(add2(lf.tgrg, L.tgrg), rt.tgrg);
  HYrg0[1] = fma2(rt.tgrg, rt.tgrg, fma2(L.tgrg, L.tgrg, mul2(lf.tgrg, lf.tgrg)));
  HYb0[0] = lf.tgb + L.tgb + rt.tgb;
  HYb0[1] = fmaf(rt.tgb, rt.tgb, fmaf(L.tgb, L.tgb, lf.tgb * lf.tgb));
#pragma unroll
  for (int s = 0; s < 3; ++s) {
    const P2 yl = (s < 2) ? lf.tgrg : bc(lf.tgb), yc = (s < 2) ? L.tgrg : bc(L.tgb), yr = (s < 2) ? rt.tgrg : bc(rt.tgb);
    const P2 xl = lf.pr[s], xc = L.pr[s], xr = rt.pr[s];
    H0[s][0] = add2(add2(xl, xc), xr);
    H0[s][1] = fma2(xr, xr, fma2(xc, xc, mul2(xl, xl)));
    H0[s][2] = fma2(xr, yr, fma2(xc, yc, mul2(xl, yl)));
  }
  const bool own = L.colok && yw >= y0 && yw < y1 && lane >= lane_lo && lane <= lane_hi;
  if (own) {
    const size_t plane = (size_t)P.H * P.W;
    P2 S[3];
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      S[s] = bc(0.f);
      if (!NOSSIM) {
        const P2 vy0 = (s < 2) ? add2(L.HYrg2[0], HYrg0[0]) : bc(L.HYb2[0] + HYb0[0]);
        const P2 vy1 = (s < 2) ? add2(L.HYrg2[1], HYrg0[1]) : bc(L.HYb2[1] + HYb0[1]);
        S[s] = ssim_window2(add2(L.H2[s][0], H0[s][0]), add2(L.H2[s][1], H0[s][1]), add2(L.H2[s][2], H0[s][2]), vy0, vy1, nullptr);
      }
    }
    const P2 e0 = sub2(L.tgrg1, L.pr1[0]), e1 = sub2(L.tgrg1, L.pr1[1]), e2 = sub2(bc(L.tgb1), L.pr1[2]);
    const float ss0 = ((0.f + S[0].x) + S[0].y) + S[2].x, ss1 = ((0.f + S[1].x) + S[1].y) + S[2].y;
    const float l10 = ((0.f + fabsf(e0.x)) + fabsf(e0.y)) + fabsf(e2.x);
    const float l11 = ((0.f + fabsf(e1.x)) + fabsf(e1.y)) + fabsf(e2.y);
    float* o = P.idloss + ((size_t)b * 2) * plane + (size_t)yw * P.W + L.xi;
    o[0] = NOSSIM ? l10 * (1.0f / 3.0f) : fmaf(0.85f / 3.0f, ss0, (0.15f / 3.0f) * l10);
    o[plane] = NOSSIM ? l11 * (1.0f / 3.0f) : fmaf(0.85f / 3.0f, ss1, (0.15f / 3.0f) * l11);
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    L.HYrg2[k] = add2(L.HYrg1[k], HYrg0[k]); L.HYrg1[k] = HYrg0[k];
    L.HYb2[k] = L.HYb1[k] + HYb0[k]; L.HYb1[k] = HYb0[k];
  }
  L.tgrg1 = L.tgrg; L.tgb1 = L.tgb;
#pragma unroll
  for (int s = 0; s < 3; ++s) {
#pragma unroll
    for (int k = 0; k < 3; ++k) { L.H2[s][k] = add2(L.H1[s][k], H0[s][k]); L.H1[s][k] = H0[s][k]; }
    L.pr1[s] = L.pr[s];
  }
}

}  // namespace md2

#endif  // __CUDACC__
