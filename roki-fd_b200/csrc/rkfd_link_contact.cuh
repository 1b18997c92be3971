/* rkfd_link_contact.cuh - net contact wrench on links from the last committing evaluation (rkFDBatchGetLinkContactWrench).
 *
 * What the committing evaluation pushed onto a link's wrench (rkFDContactForcePushWrench, rkfd_util.c:268-282; the oracle's
 * ork_lw::wext), rebuilt from its contact forces (the cf rows) and the link frames of the committed q (kin_walk of rkfd_kin.cuh
 * over the frame columns of the table):
 *   - a vertex slot of a cell on the link: +f at the vertex.  An elastic slot whose force points into the surface
 *     (dot(f, n) < 0) was written to cf but never applied (Core::contacts, Core::contacts_moving): it is left out, with the normal
 *     n of the box face closest to the vertex, chosen as Core::box_face chooses it;
 *   - the box of a moving pair on the link: -f at the vertex of the other link (the partner's reaction);
 *   - a Volume box pair: its force, and its torque about the volume centre shifted to the link origin.
 * Inactive slots hold zero forces.  The torque is taken about the link origin, force and torque in world axes.
 *
 * Compiled by nvcc into rkfd_link_contact_wrench_kernel (rkfd_engine.cu) and by g++ beside the host harness
 * (tests/link_contact/hostsim_link_contact.cpp), so that the arithmetic is checked against the oracle without a device. */
#ifndef RKFD_LINK_CONTACT_CUH
#define RKFD_LINK_CONTACT_CUH

#include "rkfd_kin.cuh"

namespace rkfd {

/* F.fr(col, c): frame column `col` as kin_walk wrote it (c < 9: R row-major, then p); C.f(slot, a): component a of the
 * slot's contact force; O.w(k, c): output column k (c < 3: force, then torque about the link origin); vert: the model's
 * vertex coordinates (ModelDev::vert) */
template <class Fr, class Cf, class Out>
RKFD_HD void link_contact_reduce(const LcwDev &t, const double *vert, const Fr &F, const Cf &C, Out &O)
{
  for(int k=0;k<t.nsel;k++) if( t.first[k] == k ) for(int c=0;c<6;c++) O.w(k,c) = 0.0;
  auto frame = [&](int col, M3 &R, V3 &p){
    R.xx = F.fr(col,0); R.xy = F.fr(col,1); R.xz = F.fr(col,2); R.yx = F.fr(col,3); R.yy = F.fr(col,4); R.yz = F.fr(col,5);
    R.zx = F.fr(col,6); R.zy = F.fr(col,7); R.zz = F.fr(col,8); p = v3(F.fr(col,9), F.fr(col,10), F.fr(col,11));
  };
  for(int j=0;j<t.nterm;j++){
    const LcwTermDev &e = t.term[j];
    M3 Rv; V3 pv; frame(e.vcol, Rv, pv);
    M3 Ro; V3 po; frame(t.ocol[e.acc], Ro, po);
    V3 fs = v3(0,0,0), ts = v3(0,0,0);
    if( e.kind == LCW_VOL ){
      const V3 f = v3(C.f(e.sofs,0), C.f(e.sofs,1), C.f(e.sofs,2)), tc = v3(C.f(e.sofs+1,0), C.f(e.sofs+1,1), C.f(e.sofs+1,2));
      const V3 cen = v3(C.f(e.sofs+2,0), C.f(e.sofs+2,1), C.f(e.sofs+2,2));
      fs = f; ts = tc + cross(cen - po, f);
    } else {
      const LcwBoxDev &bx = t.box[e.box];
      M3 Rb; V3 pb;
      Rb.xx=bx.R[0]; Rb.xy=bx.R[1]; Rb.xz=bx.R[2]; Rb.yx=bx.R[3]; Rb.yy=bx.R[4]; Rb.yz=bx.R[5]; Rb.zx=bx.R[6]; Rb.zy=bx.R[7]; Rb.zz=bx.R[8];
      pb = v3(bx.p[0], bx.p[1], bx.p[2]);
      if( bx.col >= 0 ){ M3 Rl; V3 pl; frame(bx.col, Rl, pl); pb = pl + mul(Rl, pb); Rb = mm(Rl, Rb); }   /* as Core::contacts_moving */
      for(int k=0;k<e.nvert;k++){
        const int s = e.sofs + k, vi = e.vofs + k;
        V3 f = v3(C.f(s,0), C.f(s,1), C.f(s,2));
        if( f.x == 0.0 && f.y == 0.0 && f.z == 0.0 ) continue;
        const V3 vw = pv + mul(Rv, v3(vert[3*vi], vert[3*vi+1], vert[3*vi+2]));
        if( e.elastic ){
          /* Core::box_face: the first face of least depth, outward */
          const V3 vb = tmul(Rb, vw - pb);
          const double dx = bx.half[0]-fabs(vb.x), dy = bx.half[1]-fabs(vb.y), dz = bx.half[2]-fabs(vb.z);
          int amin = 0; double dmin = dx;
          if( dy < dmin ){ dmin = dy; amin = 1; }
          if( dz < dmin ){ amin = 2; }
          const double vba = amin==0 ? vb.x : ( amin==1 ? vb.y : vb.z );
          const V3 n = ( vba >= 0 ? 1.0 : -1.0 )*( amin==0 ? col0(Rb) : ( amin==1 ? col1(Rb) : col2(Rb) ) );
          if( dot(f, n) < 0.0 ) continue;            /* computed, not applied */
        }
        if( e.kind == LCW_BOX ) f = v3(-f.x, -f.y, -f.z);
        fs = fs + f; ts = ts + cross(vw - po, f);
      }
    }
    O.w(e.acc,0) += fs.x; O.w(e.acc,1) += fs.y; O.w(e.acc,2) += fs.z;
    O.w(e.acc,3) += ts.x; O.w(e.acc,4) += ts.y; O.w(e.acc,5) += ts.z;
  }
  for(int k=0;k<t.nsel;k++) if( t.first[k] != k ) for(int c=0;c<6;c++) O.w(k,c) = O.w(t.first[k],c);
}

}  // namespace rkfd
#endif
