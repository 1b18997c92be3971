/* rkfd_math.cuh - register-resident 3-D / 6-D helpers for the fused step kernel.
 * Everything is fp64 and fully unrolled by construction (named members, no indexed arrays) so that
 * nothing is demoted to local memory. */
#ifndef RKFD_MATH_CUH
#define RKFD_MATH_CUH

#include <math.h>

#if defined(__CUDACC__)
#define RKFD_HD __host__ __device__ __forceinline__
#define RKFD_RARE static __host__ __device__ __noinline__     /* rare paths (multi-DoF joints): keep them out of the hot code */
#else
#define RKFD_HD inline
#define RKFD_RARE inline
#endif

namespace rkfd {

struct V3 { double x, y, z; };
struct M3 { double xx, xy, xz, yx, yy, yz, zx, zy, zz; };   /* row-major names: first index = row */
struct S3 { double xx, xy, xz, yy, yz, zz; };               /* symmetric */
struct V6 { V3 l, a; };                                      /* (linear, angular) */

RKFD_HD V3 v3(double x, double y, double z){ V3 r; r.x=x; r.y=y; r.z=z; return r; }

/* products and sums that the compiler may not contract into multiply-adds (the host build does not contract) */
RKFD_HD double mul_rn(double a, double b){
#if defined(__CUDA_ARCH__)
  return __dmul_rn(a, b);
#else
  return a*b;
#endif
}
RKFD_HD double add_rn(double a, double b){
#if defined(__CUDA_ARCH__)
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}
RKFD_HD double sub_rn(double a, double b){
#if defined(__CUDA_ARCH__)
  return __dsub_rn(a, b);
#else
  return a - b;
#endif
}
/* rigid-body inertia of a link about its origin from its mass m, centre of mass c and inertia Ic about c (link axes):
 * mc = m c and Io = Ic - m [c x]^2 = Ic + m (|c|^2 E - c c^T).  build_model fills the constant table with it and Core::pass2
 * forms per-environment values with it: the same operations in the same order, so that a link given the model's own values
 * gets the table's values bit for bit */
RKFD_HD void mass_prop_origin(double m, V3 c, const S3 &Ic, V3 &mc, S3 &Io){
  const double c2 = add_rn(add_rn(mul_rn(c.x, c.x), mul_rn(c.y, c.y)), mul_rn(c.z, c.z));
  mc.x = mul_rn(m, c.x); mc.y = mul_rn(m, c.y); mc.z = mul_rn(m, c.z);
  Io.xx = add_rn(Ic.xx, mul_rn(m, sub_rn(c2, mul_rn(c.x, c.x))));
  Io.xy = add_rn(Ic.xy, mul_rn(m, sub_rn(0.0, mul_rn(c.x, c.y))));
  Io.xz = add_rn(Ic.xz, mul_rn(m, sub_rn(0.0, mul_rn(c.x, c.z))));
  Io.yy = add_rn(Ic.yy, mul_rn(m, sub_rn(c2, mul_rn(c.y, c.y))));
  Io.yz = add_rn(Ic.yz, mul_rn(m, sub_rn(0.0, mul_rn(c.y, c.z))));
  Io.zz = add_rn(Ic.zz, mul_rn(m, sub_rn(c2, mul_rn(c.z, c.z))));
}
RKFD_HD V3 operator+(V3 a, V3 b){ return v3(a.x+b.x, a.y+b.y, a.z+b.z); }
RKFD_HD V3 operator-(V3 a, V3 b){ return v3(a.x-b.x, a.y-b.y, a.z-b.z); }
RKFD_HD V3 operator-(V3 a){ return v3(-a.x,-a.y,-a.z); }
RKFD_HD V3 operator*(double k, V3 a){ return v3(k*a.x, k*a.y, k*a.z); }
RKFD_HD double dot(V3 a, V3 b){ return a.x*b.x + a.y*b.y + a.z*b.z; }
RKFD_HD V3 cross(V3 a, V3 b){ return v3(a.y*b.z-a.z*b.y, a.z*b.x-a.x*b.z, a.x*b.y-a.y*b.x); }
RKFD_HD double norm(V3 a){ return sqrt(dot(a,a)); }

RKFD_HD V3 mul(const M3 &m, V3 v){ return v3(m.xx*v.x+m.xy*v.y+m.xz*v.z, m.yx*v.x+m.yy*v.y+m.yz*v.z, m.zx*v.x+m.zy*v.y+m.zz*v.z); }
RKFD_HD V3 tmul(const M3 &m, V3 v){ return v3(m.xx*v.x+m.yx*v.y+m.zx*v.z, m.xy*v.x+m.yy*v.y+m.zy*v.z, m.xz*v.x+m.yz*v.y+m.zz*v.z); }
RKFD_HD V3 mul(const S3 &m, V3 v){ return v3(m.xx*v.x+m.xy*v.y+m.xz*v.z, m.xy*v.x+m.yy*v.y+m.yz*v.z, m.xz*v.x+m.yz*v.y+m.zz*v.z); }
RKFD_HD V3 col0(const M3 &m){ return v3(m.xx,m.yx,m.zx); }
RKFD_HD V3 col1(const M3 &m){ return v3(m.xy,m.yy,m.zy); }
RKFD_HD V3 col2(const M3 &m){ return v3(m.xz,m.yz,m.zz); }
RKFD_HD M3 from_cols(V3 a, V3 b, V3 c){ M3 m; m.xx=a.x; m.yx=a.y; m.zx=a.z; m.xy=b.x; m.yy=b.y; m.zy=b.z; m.xz=c.x; m.yz=c.y; m.zz=c.z; return m; }
RKFD_HD M3 ident3(){ M3 m; m.xx=1; m.xy=0; m.xz=0; m.yx=0; m.yy=1; m.yz=0; m.zx=0; m.zy=0; m.zz=1; return m; }
RKFD_HD M3 transpose(const M3 &a){ M3 m; m.xx=a.xx; m.xy=a.yx; m.xz=a.zx; m.yx=a.xy; m.yy=a.yy; m.yz=a.zy; m.zx=a.xz; m.zy=a.yz; m.zz=a.zz; return m; }
RKFD_HD M3 mm(const M3 &a, const M3 &b){
  M3 m;
  m.xx=a.xx*b.xx+a.xy*b.yx+a.xz*b.zx; m.xy=a.xx*b.xy+a.xy*b.yy+a.xz*b.zy; m.xz=a.xx*b.xz+a.xy*b.yz+a.xz*b.zz;
  m.yx=a.yx*b.xx+a.yy*b.yx+a.yz*b.zx; m.yy=a.yx*b.xy+a.yy*b.yy+a.yz*b.zy; m.yz=a.yx*b.xz+a.yy*b.yz+a.yz*b.zz;
  m.zx=a.zx*b.xx+a.zy*b.yx+a.zz*b.zx; m.zy=a.zx*b.xy+a.zy*b.yy+a.zz*b.zy; m.zz=a.zx*b.xz+a.zy*b.yz+a.zz*b.zz;
  return m; }
/* a^T b */
RKFD_HD M3 tmm(const M3 &a, const M3 &b){ return mm(transpose(a), b); }
RKFD_HD M3 ms(const M3 &a, const S3 &b){
  M3 m;
  m.xx=a.xx*b.xx+a.xy*b.xy+a.xz*b.xz; m.xy=a.xx*b.xy+a.xy*b.yy+a.xz*b.yz; m.xz=a.xx*b.xz+a.xy*b.yz+a.xz*b.zz;
  m.yx=a.yx*b.xx+a.yy*b.xy+a.yz*b.xz; m.yy=a.yx*b.xy+a.yy*b.yy+a.yz*b.yz; m.yz=a.yx*b.xz+a.yy*b.yz+a.yz*b.zz;
  m.zx=a.zx*b.xx+a.zy*b.xy+a.zz*b.xz; m.zy=a.zx*b.xy+a.zy*b.yy+a.zz*b.yz; m.zz=a.zx*b.xz+a.zy*b.yz+a.zz*b.zz;
  return m; }
/* R A R^T for symmetric A (only the 6 distinct entries of the result) */
RKFD_HD S3 rot_sym(const M3 &R, const S3 &A){
  M3 t = ms(R, A); S3 s;
  s.xx=t.xx*R.xx+t.xy*R.xy+t.xz*R.xz; s.xy=t.xx*R.yx+t.xy*R.yy+t.xz*R.yz; s.xz=t.xx*R.zx+t.xy*R.zy+t.xz*R.zz;
  s.yy=t.yx*R.yx+t.yy*R.yy+t.yz*R.yz; s.yz=t.yx*R.zx+t.yy*R.zy+t.yz*R.zz;
  s.zz=t.zx*R.zx+t.zy*R.zy+t.zz*R.zz;
  return s; }
/* R B R^T for general B */
RKFD_HD M3 rot_gen(const M3 &R, const M3 &B){ return mm(mm(R,B), transpose(R)); }
/* [p x] M  (rows of the result are cross products of p with the columns of M) */
RKFD_HD M3 skew_mul(V3 p, const M3 &m){ return from_cols(cross(p,col0(m)), cross(p,col1(m)), cross(p,col2(m))); }
/* M [p x] : column j = M (p x e_j) */
RKFD_HD M3 mul_skew(const S3 &m, V3 p){     /* written out: products with the zero entries of [p x] are not folded by the compiler */
  M3 r;
  r.xx = m.xy*p.z - m.xz*p.y; r.yx = m.yy*p.z - m.yz*p.y; r.zx = m.yz*p.z - m.zz*p.y;
  r.xy = m.xz*p.x - m.xx*p.z; r.yy = m.yz*p.x - m.xy*p.z; r.zy = m.zz*p.x - m.xz*p.z;
  r.xz = m.xx*p.y - m.xy*p.x; r.yz = m.xy*p.y - m.yy*p.x; r.zz = m.xz*p.y - m.yz*p.x;
  return r; }

/* ---- accumulate forms: acc + M v, acc + a x b, ... as explicit fused multiply-add chains.  `acc + mul(M, v)` costs
 * four instructions per component (the compiler may not re-associate the sum), these cost three (two for a cross
 * product component): about one fp64 instruction in eight of the dynamics passes. */
RKFD_HD V3 madd(V3 a, const M3 &m, V3 v){ return v3(fma(m.xz,v.z,fma(m.xy,v.y,fma(m.xx,v.x,a.x))), fma(m.yz,v.z,fma(m.yy,v.y,fma(m.yx,v.x,a.y))), fma(m.zz,v.z,fma(m.zy,v.y,fma(m.zx,v.x,a.z)))); }
RKFD_HD V3 maddt(V3 a, const M3 &m, V3 v){ return v3(fma(m.zx,v.z,fma(m.yx,v.y,fma(m.xx,v.x,a.x))), fma(m.zy,v.z,fma(m.yy,v.y,fma(m.xy,v.x,a.y))), fma(m.zz,v.z,fma(m.yz,v.y,fma(m.xz,v.x,a.z)))); }
RKFD_HD V3 madd(V3 a, const S3 &m, V3 v){ return v3(fma(m.xz,v.z,fma(m.xy,v.y,fma(m.xx,v.x,a.x))), fma(m.yz,v.z,fma(m.yy,v.y,fma(m.xy,v.x,a.y))), fma(m.zz,v.z,fma(m.yz,v.y,fma(m.xz,v.x,a.z)))); }
RKFD_HD V3 cadd(V3 a, V3 b, V3 c){ return v3(fma(b.y,c.z,fma(-b.z,c.y,a.x)), fma(b.z,c.x,fma(-b.x,c.z,a.y)), fma(b.x,c.y,fma(-b.y,c.x,a.z))); }   /* a + b x c */
RKFD_HD V3 vfma(double k, V3 b, V3 a){ return v3(fma(k,b.x,a.x), fma(k,b.y,a.y), fma(k,b.z,a.z)); }                                        /* a + k b */
/* Br - Ar [p x]   and   Cr + [p x] Bp + ([p x] Br)^T  (shift of an articulated inertia by p, blocks of the congruence) */
RKFD_HD M3 shift_B(const M3 &Br, const S3 &A, V3 p){
  M3 r;
  r.xx = fma(A.xz,p.y,fma(-A.xy,p.z,Br.xx)); r.yx = fma(A.yz,p.y,fma(-A.yy,p.z,Br.yx)); r.zx = fma(A.zz,p.y,fma(-A.yz,p.z,Br.zx));
  r.xy = fma(A.xx,p.z,fma(-A.xz,p.x,Br.xy)); r.yy = fma(A.xy,p.z,fma(-A.yz,p.x,Br.yy)); r.zy = fma(A.xz,p.z,fma(-A.zz,p.x,Br.zy));
  r.xz = fma(A.xy,p.x,fma(-A.xx,p.y,Br.xz)); r.yz = fma(A.yy,p.x,fma(-A.xy,p.y,Br.yz)); r.zz = fma(A.yz,p.x,fma(-A.xz,p.y,Br.zz));
  return r; }
RKFD_HD S3 shift_C(const S3 &Cr, const M3 &Bp, const M3 &Br, V3 p){
  S3 r;       /* ([p x] M)_ij = (p x col_j(M))_i */
  r.xx = fma(p.y,Br.zx,fma(-p.z,Br.yx,fma(p.y,Bp.zx,fma(-p.z,Bp.yx,Cr.xx))));
  r.xy = fma(p.z,Br.xx,fma(-p.x,Br.zx,fma(p.y,Bp.zy,fma(-p.z,Bp.yy,Cr.xy))));
  r.xz = fma(p.x,Br.yx,fma(-p.y,Br.xx,fma(p.y,Bp.zz,fma(-p.z,Bp.yz,Cr.xz))));
  r.yy = fma(p.z,Br.xy,fma(-p.x,Br.zy,fma(p.z,Bp.xy,fma(-p.x,Bp.zy,Cr.yy))));
  r.yz = fma(p.x,Br.yy,fma(-p.y,Br.xy,fma(p.z,Bp.xz,fma(-p.x,Bp.zz,Cr.yz))));
  r.zz = fma(p.x,Br.yz,fma(-p.y,Br.xz,fma(p.x,Bp.yz,fma(-p.y,Bp.xz,Cr.zz))));
  return r; }

/* the same with the frame offset p of a link, short forms when p = (0,0,p.z) (x.pz) */
struct XF;
RKFD_HD V3 cadd_p(V3 a, V3 b, V3 p, int pz){ return pz ? v3(fma(b.y,p.z,a.x), fma(-b.x,p.z,a.y), a.z) : cadd(a, b, p); }          /* a + b x p */
RKFD_HD V3 padd_c(V3 a, V3 p, V3 c, int pz){ return pz ? v3(fma(-p.z,c.y,a.x), fma(p.z,c.x,a.y), a.z) : cadd(a, p, c); }           /* a + p x c */
RKFD_HD V3 madd_p(V3 a, const M3 &m, V3 p, int pz){ return pz ? v3(fma(m.xz,p.z,a.x), fma(m.yz,p.z,a.y), fma(m.zz,p.z,a.z)) : madd(a, m, p); }
RKFD_HD M3 shift_B_p(const M3 &Br, const S3 &A, V3 p, int pz){
  if( !pz ) return shift_B(Br, A, p);
  M3 r;
  r.xx = fma(-A.xy,p.z,Br.xx); r.yx = fma(-A.yy,p.z,Br.yx); r.zx = fma(-A.yz,p.z,Br.zx);
  r.xy = fma(A.xx,p.z,Br.xy);  r.yy = fma(A.xy,p.z,Br.yy);  r.zy = fma(A.xz,p.z,Br.zy);
  r.xz = Br.xz; r.yz = Br.yz; r.zz = Br.zz;
  return r; }
RKFD_HD S3 shift_C_p(const S3 &Cr, const M3 &Bp, const M3 &Br, V3 p, int pz){
  if( !pz ) return shift_C(Cr, Bp, Br, p);
  S3 r;
  r.xx = fma(-p.z,Br.yx,fma(-p.z,Bp.yx,Cr.xx));
  r.xy = fma(p.z,Br.xx,fma(-p.z,Bp.yy,Cr.xy));
  r.xz = fma(-p.z,Bp.yz,Cr.xz);
  r.yy = fma(p.z,Br.xy,fma(p.z,Bp.xy,Cr.yy));
  r.yz = fma(p.z,Bp.xz,Cr.yz);
  r.zz = Cr.zz;
  return r; }

/* ---- structured link transforms ------------------------------------------------------------------
 * A revolute link frame is R = Ro * Rz(q).  When the constant part Ro is the identity or a quarter turn
 * about x (DH alpha in {0, +90, -90} deg: the usual case), products with R are a planar rotation plus a
 * signed permutation instead of dense 3x3 products.  Everything else uses the dense path. */
enum RoClass : int { RO_GENERAL = 0, RO_IDENT = 1, RO_RXP = 2 /* Rx(+90): (x,y,z)->(x,-z,y) */, RO_RXM = 3 /* Rx(-90): (x,y,z)->(x,z,-y) */,
                     RO_RXS = 4 /* Rx(sg*90), sign sg = +-1 read from the link table at run time (rolled link loops) */ };
/* sign of the quarter turn: a literal for RXP / RXM (multiplications by it fold away), the table value for RXS */
RKFD_HD double ro_sign(int cls, double table_sg){ return cls == RO_RXP ? 1.0 : ( cls == RO_RXM ? -1.0 : table_sg ); }

RKFD_HD V3 rz_mul(double c, double s, V3 v){ return v3(c*v.x - s*v.y, s*v.x + c*v.y, v.z); }
RKFD_HD V3 rz_tmul(double c, double s, V3 v){ return v3(c*v.x + s*v.y, c*v.y - s*v.x, v.z); }
/* Rz A Rz^T, A symmetric */
RKFD_HD S3 rz_sym(double c, double s, const S3 &A){
  const double txx = c*A.xx - s*A.xy, txy = c*A.xy - s*A.yy, tyx = s*A.xx + c*A.xy, tyy = s*A.xy + c*A.yy;
  S3 r; r.xx = c*txx - s*txy; r.xy = s*txx + c*txy; r.yy = s*tyx + c*tyy;
  r.xz = c*A.xz - s*A.yz; r.yz = s*A.xz + c*A.yz; r.zz = A.zz; return r; }
/* Rz B Rz^T, B general */
RKFD_HD M3 rz_gen(double c, double s, const M3 &B){
  const double txx = c*B.xx - s*B.yx, txy = c*B.xy - s*B.yy, txz = c*B.xz - s*B.yz;
  const double tyx = s*B.xx + c*B.yx, tyy = s*B.xy + c*B.yy, tyz = s*B.xz + c*B.yz;
  M3 r;
  r.xx = c*txx - s*txy; r.xy = s*txx + c*txy; r.xz = txz;
  r.yx = c*tyx - s*tyy; r.yy = s*tyx + c*tyy; r.yz = tyz;
  r.zx = c*B.zx - s*B.zy; r.zy = s*B.zx + c*B.zy; r.zz = B.zz; return r; }
/* Ro v, Ro^T v, Ro A Ro^T, Ro B Ro^T, M Ro for the special classes (cls != RO_GENERAL) */
RKFD_HD V3 ro_mul(int cls, double sg, V3 v){ return cls == RO_IDENT ? v : v3(v.x, -sg*v.z, sg*v.y); }
RKFD_HD V3 ro_tmul(int cls, double sg, V3 v){ return cls == RO_IDENT ? v : v3(v.x, sg*v.z, -sg*v.y); }
RKFD_HD S3 ro_sym(int cls, double sg, const S3 &A){
  if( cls == RO_IDENT ) return A;
  S3 r;                                                /* rows: x<-x, y<- -sg z, z<- sg y */ r.xx = A.xx; r.xy = -sg*A.xz; r.xz = sg*A.xy; r.yy = A.zz; r.yz = -A.yz; r.zz = A.yy; return r; }
RKFD_HD M3 ro_gen(int cls, double sg, const M3 &B){
  if( cls == RO_IDENT ) return B;
  M3 r;
  r.xx = B.xx;     r.xy = -sg*B.xz; r.xz = sg*B.xy;
  r.yx = -sg*B.zx; r.yy = B.zz;     r.yz = -B.zy;
  r.zx = sg*B.yx;  r.zy = -B.yz;    r.zz = B.yy; return r; }
/* M Ro: columns of the result are M applied to the columns of Ro */
RKFD_HD M3 mul_ro(int cls, double sg, const M3 &M){
  if( cls == RO_IDENT ) return M;                     /* Ro columns: e_x, sg e_z, -sg e_y */
  return from_cols(col0(M), sg*col2(M), (-sg)*col1(M)); }

/* link frame w.r.t. its parent */
struct XF {
  int fast;        /* 1: R = Ro(cls) * Rz(c,s) handled structurally; 0: dense R */
  int cls;
  double sg;       /* sign of the quarter turn (fast, cls != RO_IDENT) */
  double c, s;
  M3 R;            /* dense rotation (fast == 0) */
  V3 p;            /* origin of the link frame in parent coordinates */
  int pz;          /* p = (0, 0, p.z): the link origin sits on the parent's z axis (warp-uniform, from the table) - the
                      products with [p x] then lose two thirds of their terms */
  V3 ptl;          /* R^T p */
};
RKFD_HD V3 xf_tmul(const XF &x, V3 v){ return x.fast ? rz_tmul(x.c, x.s, ro_tmul(x.cls, x.sg, v)) : tmul(x.R, v); }
RKFD_HD V3 xf_mul(const XF &x, V3 v){ return x.fast ? ro_mul(x.cls, x.sg, rz_mul(x.c, x.s, v)) : mul(x.R, v); }
RKFD_HD S3 xf_sym(const XF &x, const S3 &A){ return x.fast ? ro_sym(x.cls, x.sg, rz_sym(x.c, x.s, A)) : rot_sym(x.R, A); }
RKFD_HD M3 xf_gen(const XF &x, const M3 &B){ return x.fast ? ro_gen(x.cls, x.sg, rz_gen(x.c, x.s, B)) : rot_gen(x.R, B); }
/* Rw R */
RKFD_HD M3 xf_world(const XF &x, const M3 &Rw){
  if( !x.fast ) return mm(Rw, x.R);
  const M3 T = mul_ro(x.cls, x.sg, Rw); const V3 t0 = col0(T), t1 = col1(T);
  return from_cols(x.c*t0 + x.s*t1, x.c*t1 - x.s*t0, col2(T)); }

/* angle-axis vector -> rotation matrix (Rodrigues) */
RKFD_RARE M3 aa_to_mat(V3 aa){
  double th2 = dot(aa,aa), A, B;
  if( th2 < 1.0e-24 ){ A = 1.0; B = 0.5; }
  else { double th = sqrt(th2); A = sin(th)/th; B = (1.0-cos(th))/th2; }
  /* R = I + A K + B K^2, K = [aa x] ; K^2 = aa aa^T - th2 I */
  M3 m;
  m.xx = 1.0 + B*(aa.x*aa.x - th2); m.yy = 1.0 + B*(aa.y*aa.y - th2); m.zz = 1.0 + B*(aa.z*aa.z - th2);
  m.xy = -A*aa.z + B*aa.x*aa.y; m.yx =  A*aa.z + B*aa.x*aa.y;
  m.xz =  A*aa.y + B*aa.x*aa.z; m.zx = -A*aa.y + B*aa.x*aa.z;
  m.yz = -A*aa.x + B*aa.y*aa.z; m.zy =  A*aa.x + B*aa.y*aa.z;
  return m; }

/* aa <- log( R(w) R(aa) ) through unit quaternions */
RKFD_RARE V3 aa_cascade(V3 aa, V3 w){
  double th, s, q10, q20; V3 q1, q2;
  if( w.x == 0.0 && w.y == 0.0 && w.z == 0.0 ) return aa;      /* no increment: the displacement is kept bit for bit (a held joint) */
  th = norm(aa);
  if( th < 1.0e-12 ){ q10 = 1.0; q1 = 0.5*aa; } else { s = sin(0.5*th)/th; q10 = cos(0.5*th); q1 = s*aa; }
  th = norm(w);
  if( th < 1.0e-12 ){ q20 = 1.0; q2 = 0.5*w; } else { s = sin(0.5*th)/th; q20 = cos(0.5*th); q2 = s*w; }
  double q0 = q20*q10 - q2.x*q1.x - q2.y*q1.y - q2.z*q1.z;
  V3 q = v3( q20*q1.x + q2.x*q10 + q2.y*q1.z - q2.z*q1.y,
             q20*q1.y - q2.x*q1.z + q2.y*q10 + q2.z*q1.x,
             q20*q1.z + q2.x*q1.y - q2.y*q1.x + q2.z*q10 );
  if( q0 < 0 ){ q0 = -q0; q = -q; }
  double n = norm(q);
  if( n < 1.0e-12 ) return 2.0*q;
  th = 2.0*atan2(n,q0);
  return (th/n)*q; }

}  // namespace rkfd
#endif
