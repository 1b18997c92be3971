/* rkfd_kin.cuh - world frames and velocities of links from the committed state (rkFDBatchGetLinkFrames).
 *
 * The joint model is the one of pass 1 of the step kernel (Core::pass1_link in rkfd_core.cuh) without its scratch stores and
 * contacts: the same rkfd_math.cuh transforms, the same products in the same order.  Revolute sin/cos come from sincos(q) (the
 * "fresh" path of Core::revol_state), so the frames agree with the step kernel's internal ones to rounding.  A breakable-float
 * joint contributes its displacement always and its joint velocity only once broken (pivot bit of its first dof), as in pass 1.
 *
 * Compiled by nvcc into the engine's kinematics kernel (rkfd_engine.cu) and by g++ into the host harness
 * (tests/hostsim/kin_harness.cpp), so that the arithmetic is checked against the oracle without a device.  The table is a KinDev (rkfd_types.h, kin_table in
 * rkfd_model.cpp). */
#ifndef RKFD_KIN_CUH
#define RKFD_KIN_CUH

#include "rkfd_math.cuh"
#include "rkfd_types.h"

#if defined(__CUDA_ARCH__)
#define RKFD_KIN_CTZ(x) (__ffs(x) - 1)
#else
#define RKFD_KIN_CTZ(x) __builtin_ctz(x)
#endif

namespace rkfd {

/* frame of a link w.r.t. its parent (x) and joint velocity in link axes (vJ linear, wJ angular).  `J` gives the joint's values:
 * J.q(k), J.qd(k) for dof k of the joint.  vel = false: the joint velocity is not formed.  brk: a breakable-float joint has
 * broken */
template <class Jv>
RKFD_HD void kin_joint(const KinLinkDev &L, const Jv &J, bool vel, bool brk, XF &x, V3 &vJ, V3 &wJ)
{
  M3 Ro; Ro.xx=L.Ro[0]; Ro.xy=L.Ro[1]; Ro.xz=L.Ro[2]; Ro.yx=L.Ro[3]; Ro.yy=L.Ro[4]; Ro.yz=L.Ro[5]; Ro.zx=L.Ro[6]; Ro.zy=L.Ro[7]; Ro.zz=L.Ro[8];
  const V3 po = v3(L.po[0], L.po[1], L.po[2]);
  x.fast = 0; x.cls = L.cls; x.sg = L.sg; x.c = 1.0; x.s = 0.0; x.pz = L.pz;
  vJ = v3(0,0,0); wJ = v3(0,0,0);
  switch(L.jtype){
  case J_REVOL: {
    double sn, co; sincos(J.q(0), &sn, &co);
    x.s = sn; x.c = co; x.p = po;
    if( L.cls != RO_GENERAL ) x.fast = 1;
    else { const V3 o0 = col0(Ro), o1 = col1(Ro); x.R = from_cols(co*o0 + sn*o1, co*o1 - sn*o0, col2(Ro)); }
    if( vel ) wJ.z = J.qd(0);
  } break;
  case J_PRISM: x.R = Ro; x.p = po + J.q(0)*col2(Ro); if( vel ) vJ.z = J.qd(0); break;
  case J_SPHER:
    x.R = mm(Ro, aa_to_mat(v3(J.q(0), J.q(1), J.q(2)))); x.p = po;
    if( vel ) wJ = tmul(x.R, mul(Ro, v3(J.qd(0), J.qd(1), J.qd(2))));
    break;
  case J_FLOAT: case J_BRFLOAT:
    x.R = mm(Ro, aa_to_mat(v3(J.q(3), J.q(4), J.q(5)))); x.p = po + mul(Ro, v3(J.q(0), J.q(1), J.q(2)));
    if( vel && ( L.jtype == J_FLOAT || brk ) ){
      vJ = tmul(x.R, mul(Ro, v3(J.qd(0), J.qd(1), J.qd(2)))); wJ = tmul(x.R, mul(Ro, v3(J.qd(3), J.qd(4), J.qd(5)))); }
    break;
  case J_CYLIN: {
    double s1, c1; sincos(J.q(1), &s1, &c1);
    const V3 o0 = col0(Ro), o1 = col1(Ro);
    x.R = from_cols(c1*o0 + s1*o1, c1*o1 - s1*o0, col2(Ro)); x.p = po + J.q(0)*col2(Ro);
    if( vel ){ vJ.z = J.qd(0); wJ.z = J.qd(1); }
  } break;
  case J_HOOKE: {
    double s0, c0, s1, c1; sincos(J.q(0), &s0, &c0); sincos(J.q(1), &s1, &c1);
    M3 RJ; RJ.xx = c0*c1; RJ.xy = -s0; RJ.xz = c0*s1; RJ.yx = s0*c1; RJ.yy = c0; RJ.yz = s0*s1; RJ.zx = -s1; RJ.zy = 0.0; RJ.zz = c1;
    x.R = mm(Ro, RJ); x.p = po;
    if( vel ){ const double v0 = J.qd(0), v1 = J.qd(1); wJ = v3(-s1*v0, v1, c1*v0); }
  } break;
  default: x.R = Ro; x.p = po; break;
  }
}

/* the outward walk over t.walk.  Per visited link: the frame and velocity of its parent come from registers when the parent
 * was the link visited last, from the keep slot otherwise (roots start at the world frame at rest).
 *   S.q(k), S.qd(k): dof k of the environment; S.piv(): its pivot word (read only when t.brk)
 *   K.st(slot, c, v), K.ld(slot, c): the keep slots (KIN_KEEP doubles each)
 *   O.frame(col, c, v) (c < 12: R row-major, then p), O.vel(col, c, v) (c < 6: linear, angular in world axes)
 * wf / wv: frames / velocities are wanted. */
template <class Src, class Keep, class Out>
RKFD_HD void kin_walk(const KinDev &t, const Src &S, Keep &K, Out &O, bool wf, bool wv)
{
  const unsigned piv = t.brk ? S.piv() : 0u;
  M3 Rw = ident3(); V3 pw = v3(0,0,0), vl = v3(0,0,0), om = v3(0,0,0);
  int prev = -1;
  for(int w=0; w<t.nwalk; w++){
    const int i = t.walk[w];
    const KinLinkDev &L = t.link[i];
    if( L.parent < 0 ){ Rw = ident3(); pw = v3(0,0,0); vl = v3(0,0,0); om = v3(0,0,0); }
    else if( L.parent != prev ){
      const int s = t.link[L.parent].keep;
      Rw.xx = K.ld(s,0); Rw.xy = K.ld(s,1); Rw.xz = K.ld(s,2); Rw.yx = K.ld(s,3); Rw.yy = K.ld(s,4); Rw.yz = K.ld(s,5);
      Rw.zx = K.ld(s,6); Rw.zy = K.ld(s,7); Rw.zz = K.ld(s,8); pw = v3(K.ld(s,9), K.ld(s,10), K.ld(s,11));
      if( wv ){ vl = v3(K.ld(s,12), K.ld(s,13), K.ld(s,14)); om = v3(K.ld(s,15), K.ld(s,16), K.ld(s,17)); }
    }
    struct Jv {
      const Src &S; int o;
      RKFD_HD double q(int k) const { return S.q(o + k); }
      RKFD_HD double qd(int k) const { return S.qd(o + k); }
    } J{S, L.qofs};
    XF x; V3 vJ, wJ;
    kin_joint(L, J, wv, (piv >> L.qofs) & 1u, x, vJ, wJ);
    /* pass 1: om' = R^T om + wJ, v' = R^T (v + om x p) + vJ, pw' = pw + Rw p, Rw' = Rw R */
    if( wv ){
      const V3 vl_n = xf_tmul(x, cadd_p(vl, om, x.p, x.pz)) + vJ;
      om = xf_tmul(x, om) + wJ; vl = vl_n;
    }
    pw = madd_p(pw, Rw, x.p, x.pz); Rw = xf_world(x, Rw);
    prev = i;
    if( L.keep >= 0 ){
      const int s = L.keep;
      K.st(s,0,Rw.xx); K.st(s,1,Rw.xy); K.st(s,2,Rw.xz); K.st(s,3,Rw.yx); K.st(s,4,Rw.yy); K.st(s,5,Rw.yz);
      K.st(s,6,Rw.zx); K.st(s,7,Rw.zy); K.st(s,8,Rw.zz); K.st(s,9,pw.x); K.st(s,10,pw.y); K.st(s,11,pw.z);
      if( wv ){ K.st(s,12,vl.x); K.st(s,13,vl.y); K.st(s,14,vl.z); K.st(s,15,om.x); K.st(s,16,om.y); K.st(s,17,om.z); }
    }
    if( !L.omask ) continue;
    V3 vw = v3(0,0,0), ow = v3(0,0,0);
    if( wv ){ vw = mul(Rw, vl); ow = mul(Rw, om); }
    for(unsigned mk = L.omask; mk; mk &= mk - 1){
      const int k = RKFD_KIN_CTZ(mk);
      if( wf ){
        O.frame(k,0,Rw.xx); O.frame(k,1,Rw.xy); O.frame(k,2,Rw.xz); O.frame(k,3,Rw.yx); O.frame(k,4,Rw.yy); O.frame(k,5,Rw.yz);
        O.frame(k,6,Rw.zx); O.frame(k,7,Rw.zy); O.frame(k,8,Rw.zz); O.frame(k,9,pw.x); O.frame(k,10,pw.y); O.frame(k,11,pw.z);
      }
      if( wv ){ O.vel(k,0,vw.x); O.vel(k,1,vw.y); O.vel(k,2,vw.z); O.vel(k,3,ow.x); O.vel(k,4,ow.y); O.vel(k,5,ow.z); }
    }
  }
}

}  // namespace rkfd
#endif
