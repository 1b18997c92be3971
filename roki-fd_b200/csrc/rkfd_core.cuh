/* rkfd_core.cuh - one environment's rkFDUpdate, written once for the sm_100a kernel.
 *
 * Thread-per-environment formulation of the reference step (reference src/rkfd_sim.c:560-566):
 * 4 Runge-Kutta-Gill stage evaluations + 1 committing reference evaluation, each evaluation =
 *   pass 1 (outward)  FK + link velocities          <- _rkFDConnectJointState   rkfd_sim.c:290-302
 *                     vertex/box collision          <- _rkFDUpdateCD            rkfd_sim.c:466-471
 *                     penalty contact + Coulomb     <- rkFDSolverPenalty        rkfd_penalty.c:11-31
 *   pass 2 (inward)   joint friction / motor torque <- rkFDJointFriction        rkfd_util.c:366-387
 *                     articulated inertia + bias    <- rkChainUpdateABI [EXT]   rkfd_sim.c:509-520
 *   pass 3 (outward)  accelerations, q''            <- rkChainGetJointAccAll    rkfd_sim.c:521
 *                     RKG stage bookkeeping         <- zODE2Update [EXT]        rkfd_sim.c:562
 * The per-link quantities that must survive between passes live in a per-thread scratch column
 * (shared memory, element k of thread t at [k*BLOCK + t]: conflict-free 64-bit accesses); the
 * running articulated inertia of a serial chain segment stays in registers.
 *
 * The same source is compiled (a) by nvcc into the product kernel and (b) by g++ into a host
 * harness that only tests/ loads, to debug the arithmetic where no GPU exists.  The product
 * library contains (a) only.
 */
#ifndef RKFD_CORE_CUH
#define RKFD_CORE_CUH

#include "rkfd_types.h"
#include "rkfd_math.cuh"

#if defined(__CUDACC__)
#define RKFD_NOINLINE static __host__ __device__ __noinline__
#else
#define RKFD_NOINLINE inline
#endif
#if defined(__CUDA_ARCH__)
#define RKFD_POPC64(x) __popcll(x)
#define RKFD_FFS32(x) __ffs(x)
#define RKFD_FFS64(x) __ffsll((long long)(x))
#else
#define RKFD_POPC64(x) __builtin_popcountll(x)
#define RKFD_FFS32(x) __builtin_ffs(x)
#define RKFD_FFS64(x) __builtin_ffsll((long long)(x))
#endif

/* unroll factor of the rolled link loops (1: one body per pass) */
#ifndef RKFD_ROLL_UNROLL
#define RKFD_ROLL_UNROLL 1
#endif

namespace rkfd {

constexpr int ROLL_UNROLL = RKFD_ROLL_UNROLL;

/* scratch slots per link by joint type */
RKFD_HD int link_slot_count(int jtype, int has_rigid){
  switch(jtype){
    case J_REVOL: case J_PRISM: return has_rigid ? 16 : 10;    /* w,gd->U (6), sin, cos, Dinv, u [, w,gd (6)] */
    case J_SPHER: return has_rigid ? 42 : 36;                  /* U (18, w/gd aliased), Dinv (6), u (3), Rrel (9) [, w,gd] */
    case J_CYLIN: case J_HOOKE: return has_rigid ? 38 : 32;    /* U (12, w/gd aliased), Dinv (3), u (2), Rrel (9), prel (3), sin/cos q1 (2), pad [, w,gd] */
    case J_FLOAT: return has_rigid ? 45 : 18; /* a0 (6, w/gd aliased), Rrel (9), prel (3) [, IA^-1 (21), w,gd (6)] */
    case J_BRFLOAT: return has_rigid ? 52 : 46; /* a0 (6), Rrel (9), prel (3), IA (rigid joint) or IA^-1 (broken) (21), pA (6), broken flag [, w,gd (6)] */
    default: return 6;                        /* w, gd */
  }
}
/* offset of (w, gd) inside the link slots */
RKFD_HD int link_w_offset(int jtype, int has_rigid){
  if( !has_rigid ) return 0;
  switch(jtype){ case J_REVOL: case J_PRISM: return 10; case J_SPHER: return 36; case J_FLOAT: return 39; case J_CYLIN: case J_HOOKE: return 32; case J_BRFLOAT: return 46; default: return 0; }
}
constexpr int BRANCH_SLOTS = 15;   /* pass 1: Rw(9) pw(3) vl(3); pass 3: a(6) w(3) */
constexpr int ACCUM_SLOTS = 27;    /* A(6) B(9) C(6) pf(3) pn(3) */
constexpr int WEXT_SLOTS = 6;
constexpr int FRAME_SLOTS = 24;    /* rigid worlds, links with cells: Rw(9) pw(3) vl(3) w(3) a(6) */
constexpr int GEO_DOUBLES = 28;    /* per rigid contact: vw n t1 t2 d vel prob rl (8 x 3), slot, link, pair, partner link (-1: static) */
/* per-environment workspace of the wrench-coordinate contact paths: Lambda (6x6, column-major) per group, then per contact
 * g (3x6) h (3x6) b (3) diag (3) f (3) rho (3) prob (3) mu slot */
constexpr int MAX_RG = 4;                      /* contact groups (links in different chains) of the wrench-coordinate paths */
constexpr int W1_CT = 36*MAX_RG, W1_CTN = 53;
/* anti-cycling history of the Vert active-set loop (rkfd_opt_qp.c:152-171 keeps an unbounded list): QP_HIST entries of
 * (active sets of 3 vertices packed into one double - 16 bits each, exact - ..., objective value) */
constexpr int QP_HIST = 128;
RKFD_HD int qp_hist_stride(int nrs){ return (nrs + 2)/3 + 1; }

enum StageMode : int { ST_K1 = 0, ST_K2 = 1, ST_K3 = 2, ST_K4 = 3, ST_REF = 4, ST_EVAL = 5, ST_EVAL_REF = 6,
                       ST_PROBE = 7 /* acceleration pass of rkFDUpdateAccBias: no integrator bookkeeping, no q'' output */ };

/* symmetric 6x6 inverse through Cholesky; a is the full row-major matrix, overwritten */
RKFD_NOINLINE void spd6_inverse(double (&a)[36]){
  double L[36], Li[36];
#pragma unroll
  for(int k=0;k<36;k++){ L[k]=0; Li[k]=0; }
#pragma unroll
  for(int j=0;j<6;j++){
    double s = a[6*j+j];
#pragma unroll
    for(int k=0;k<6;k++) if(k<j) s -= L[6*j+k]*L[6*j+k];
    L[6*j+j] = sqrt(s);
    double inv = 1.0/L[6*j+j];
#pragma unroll
    for(int i=0;i<6;i++) if(i>j){
      double t = a[6*i+j];
#pragma unroll
      for(int k=0;k<6;k++) if(k<j) t -= L[6*i+k]*L[6*j+k];
      L[6*i+j] = t*inv;
    }
  }
#pragma unroll
  for(int j=0;j<6;j++){
    Li[6*j+j] = 1.0/L[6*j+j];
#pragma unroll
    for(int i=0;i<6;i++) if(i>j){
      double s = 0;
#pragma unroll
      for(int k=0;k<6;k++) if(k>=j && k<i) s -= L[6*i+k]*Li[6*k+j];
      Li[6*i+j] = s/L[6*i+i];
    }
  }
#pragma unroll
  for(int i=0;i<6;i++)
#pragma unroll
    for(int j=0;j<6;j++){
      double s = 0;
#pragma unroll
      for(int k=0;k<6;k++) if(k>=i && k>=j) s += Li[6*k+i]*Li[6*k+j];
      a[6*i+j] = s;
    }
}

/* symmetric 3x3 inverse (adjugate) */
RKFD_HD S3 sym3_inverse(const S3 &d){
  S3 c;
  c.xx = d.yy*d.zz - d.yz*d.yz; c.xy = d.xz*d.yz - d.xy*d.zz; c.xz = d.xy*d.yz - d.xz*d.yy;
  c.yy = d.xx*d.zz - d.xz*d.xz; c.yz = d.xy*d.xz - d.xx*d.yz; c.zz = d.xx*d.yy - d.xy*d.xy;
  double det = d.xx*c.xx + d.xy*c.xy + d.xz*c.xz, inv = 1.0/det;
  c.xx*=inv; c.xy*=inv; c.xz*=inv; c.yy*=inv; c.yz*=inv; c.zz*=inv;
  return c;
}

/* ---- model specialisation -------------------------------------------------------------------------
 * The generic kernel interprets the link table at run time (loop over links, switch on the joint type,
 * scratch slots read from the table).  For the common robot-arm shape - fixed base + serial revolute links
 * whose constant frame rotations are quarter turns about x or the identity, collision cells on the last link
 * only, elastic pairs only - `SpecSerialRev<NL,CLS>` makes topology, joint types, rotation classes and the
 * scratch map compile-time constants: the link loops unroll completely, every table entry becomes a
 * constant-bank operand with an immediate offset, every scratch access an LDS/STS with an immediate offset,
 * and the joint-type switches disappear.  Same arithmetic, same order of operations: results are bit-identical
 * to the generic kernel.  The host picks a compiled specialisation when the model matches (spec_match). */
/* compile-time description of one link handed to the pass bodies: joint type, rotation class, root flag;
 * -1 = not known at compile time (the Spec accessor / the link table decides) */
template <int JT_, int CLS_, int ROOT_> struct LinkTag { static constexpr int jt = JT_, cls = CLS_, root = ROOT_; };
using TagRT = LinkTag<-1, -1, -1>;

/* FUSE = 1: pass 3 of a stage and pass 1 of the next walk the links together (Core::outward) - serial arms without rigid
 * pairs, whose link i depends on link i-1 only; the generic kernel keeps the passes apart (tree worlds share branch slots
 * between pass 1 and pass 3) */
struct SpecGeneric {
  static constexpr int ID = 0, NL = 0, UNROLL = 1, NSCRATCH = 0, ROLL = 0, FUSE = 0;
  static RKFD_HD int nl(const ModelDev &m){ return m.nl; }
  static RKFD_HD int jtype(int, const LinkDev &L){ return L.jtype; }
  static RKFD_HD int parent(int, const LinkDev &L){ return L.parent; }
  static RKFD_HD int serial(int, const LinkDev &L){ return L.serial; }
  static RKFD_HD int slot(int, const LinkDev &L){ return L.slot; }
  static RKFD_HD int wslot(int, const LinkDev &L){ return L.wslot; }
  static RKFD_HD int rcls(int, const LinkDev &L){ return L.rcls; }
  static RKFD_HD int qofs(int, const LinkDev &L){ return L.qofs; }
  static RKFD_HD int ndof(int, const LinkDev &L){ return L.ndof; }
  static RKFD_HD int branch_slot(int, const LinkDev &L){ return L.branch_slot; }
  static RKFD_HD int accum_slot(int, const LinkDev &L){ return L.accum_slot; }
  static RKFD_HD int wext_slot(int, const LinkDev &L){ return L.wext_slot; }
  static RKFD_HD int frame_slot(int, const LinkDev &L){ return L.frame_slot; }
  static RKFD_HD int fext_row(int, const LinkDev &L){ return L.fext_row; }
  static RKFD_HD int rk_slot(const ModelDev &m){ return m.rk_slot; }
  static RKFD_HD int nq(const ModelDev &m){ return m.nq; }
  /* 1-DoF joints: slots of (sin, cos, 1/D, u) in the "T space" (Ctx::TL/TS) - the scratch column itself here */
  static RKFD_HD int sc(int, const LinkDev &L){ return L.sc; }
  static constexpr int TM = 0, NTSPACE = 0, SCS = 0, TCOLS = 128;
};
/* The generic table-driven kernel with the T space in tensor memory (worlds without rigid pairs; the table carries
 * the tensor-memory layout, model_layout(m, true)): trees, floating bases, any joint mix.  256 TMEM columns per
 * warpgroup = 128 doubles per thread, two 128-thread CTAs per SM. */
struct SpecGenericTM : SpecGeneric { static constexpr int ID = 11, TM = 1, TCOLS = 256; };
constexpr int SPEC_GENERIC_TM = 11, SPEC_GENERIC_TM_MAX_T = 128;
/* link 0 = fixed root, links 1..NL-1 revolute and serial; CLS: 2 bits per revolute link (RoClass 1..3) */
/* TM_ = 1: the integrator stage state and (sin, cos, 1/D, u) of every joint live in TENSOR MEMORY (tcgen05.st/ld,
 * one TMEM lane per thread, 8 bytes per element) instead of the shared-memory column, which then holds 6 doubles per
 * link + the external wrench: 54 instead of 110 doubles per environment for the 7-DoF arm -> 16 instead of 8 resident
 * warps per SM (the kernel is latency bound, profiles/).  T-space accesses are warp-collective: they only appear
 * in warp-uniform code. */
template <int ID_, int NL_, unsigned CLS_, int TM_>
struct SpecSerialRev {
  static constexpr int ID = ID_, NL = NL_, UNROLL = NL_, TM = TM_, ROLL = 0, SCS = 0, TCOLS = 128, FUSE = 1;
  static constexpr int WEXT = TM_ ? 6*NL_ : 6 + 10*(NL_-1);
  static constexpr int RK = TM_ ? 4*(NL_-1) : WEXT + 6;                 /* T space when TM_ */
  static constexpr int NSCRATCH = TM_ ? WEXT + 6 : RK + 4*(NL_-1);     /* shared-memory doubles per environment */
  static constexpr int NTSPACE = TM_ ? 8*(NL_-1) : 0;                   /* tensor-memory doubles per environment */
  static RKFD_HD int sc(int i, const LinkDev &L){ return TM_ ? 4*(i-1) : slot(i, L) + 6; }
  static RKFD_HD int nl(const ModelDev &){ return NL_; }
  static RKFD_HD int jtype(int i, const LinkDev &){ return i == 0 ? J_FIXED : J_REVOL; }
  static RKFD_HD int parent(int i, const LinkDev &){ return i - 1; }
  static RKFD_HD int serial(int i, const LinkDev &){ return i > 0 ? 1 : 0; }
  static RKFD_HD int slot(int i, const LinkDev &){ return TM_ ? 6*i : ( i == 0 ? 0 : 6 + 10*(i-1) ); }
  static RKFD_HD int wslot(int i, const LinkDev &L){ return slot(i, L); }
  static RKFD_HD int rcls(int i, const LinkDev &){ return i == 0 ? 0 : (int)((CLS_ >> (2*(i-1))) & 3u); }
  static RKFD_HD int qofs(int i, const LinkDev &){ return i > 0 ? i - 1 : 0; }
  static RKFD_HD int ndof(int i, const LinkDev &){ return i > 0 ? 1 : 0; }
  static RKFD_HD int branch_slot(int, const LinkDev &){ return -1; }
  static RKFD_HD int accum_slot(int, const LinkDev &){ return -1; }
  static RKFD_HD int wext_slot(int i, const LinkDev &L){ return ( i == NL_-1 && L.cell_end > L.cell_begin ) ? WEXT : -1; }
  static RKFD_HD int frame_slot(int, const LinkDev &){ return -1; }
  static constexpr RKFD_HD int fext_row(int, const LinkDev &){ return -1; }     /* external wrenches: generic kernels only */
  static RKFD_HD int rk_slot(const ModelDev &){ return RK; }
  static RKFD_HD int nq(const ModelDev &){ return NL_ - 1; }
};
/* Same model shape, ROLLED link loops: the base link is peeled off, the revolute links run through ONE loop body per
 * pass whose link index is a run-time (warp-uniform) value.  Every revolute frame must be a quarter turn about x; its
 * sign comes from the link table, so any pattern of +-90 degree twists shares the code.  Why: the fully unrolled
 * kernel is ~110 KB of straight-line code per evaluation, streamed through the 32 KB L1.5 / 6 KB L0 instruction caches
 * by every warp (ncu: no_instruction is its second largest stall); the rolled bodies are ~7 KB per pass and stay
 * cached.  Costs: table entries are fetched through uniform registers instead of immediate constant operands, and a
 * handful of multiplications by the sign.  Scratch layout = the tensor-memory layout of SpecSerialRev<.,.,.,1>. */
/* RG_ = 1: worlds with rigid pairs, all of them on the last link, MLCP solver (Core::rigid_mlcp_single).  Pass 2 runs
 * twice per evaluation there, so the angular velocity keeps its own 3 slots next to U, and the last
 * link publishes its world frame / velocity / acceleration (24 slots) for the contact solve. */
/* GEN_ = 1: the constant frame rotations of the revolute links are arbitrary (dense 3x3 products instead of the
 * quarter-turn forms): every fixed-base serial revolute arm gets the rolled kernel, whatever its DH twists. */
template <int ID_, int NL_, int RG_ = 0, int GEN_ = 0>
struct SpecSerialRevRolled {
  static constexpr int ID = ID_, NL = NL_, UNROLL = 1, TM = 1, ROLL = 1, RG = RG_, RCLS = GEN_ ? RO_GENERAL : RO_RXS, FUSE = !RG_;
  /* RG: (sin, cos, 1/D, u) stay in the shared-memory column (SCS): the contact solve reads them for OTHER lanes'
   * environments (lane-parallel probes) and in divergent code, which tensor memory allows neither */
  static constexpr int SCS = RG_, TCOLS = 128;
  static constexpr int PER = RG_ ? 13 : 6, FRAME = PER*NL_, WEXT = FRAME + (RG_ ? 24 : 0);
  static constexpr int RK = RG_ ? 0 : 4*(NL_-1), NSCRATCH = WEXT + 6, NTSPACE = (RG_ ? 4 : 8)*(NL_-1);
  static RKFD_HD int nl(const ModelDev &){ return NL_; }
  static RKFD_HD int jtype(int i, const LinkDev &){ return i == 0 ? J_FIXED : J_REVOL; }
  static RKFD_HD int parent(int i, const LinkDev &){ return i - 1; }
  static RKFD_HD int serial(int i, const LinkDev &){ return i > 0 ? 1 : 0; }
  static RKFD_HD int slot(int i, const LinkDev &){ return PER*i; }
  static RKFD_HD int wslot(int i, const LinkDev &){ return PER*i + (RG_ ? 6 : 0); }
  static RKFD_HD int rcls(int i, const LinkDev &){ return i == 0 ? RO_GENERAL : RCLS; }
  static RKFD_HD int qofs(int i, const LinkDev &){ return i > 0 ? i - 1 : 0; }
  static RKFD_HD int ndof(int i, const LinkDev &){ return i > 0 ? 1 : 0; }
  static RKFD_HD int branch_slot(int, const LinkDev &){ return -1; }
  static RKFD_HD int accum_slot(int, const LinkDev &){ return -1; }
  static RKFD_HD int wext_slot(int i, const LinkDev &L){ return ( i == NL_-1 && L.cell_end > L.cell_begin ) ? WEXT : -1; }
  static RKFD_HD int frame_slot(int i, const LinkDev &L){ return ( RG_ && i == NL_-1 && L.cell_end > L.cell_begin ) ? FRAME : -1; }
  static constexpr RKFD_HD int fext_row(int, const LinkDev &){ return -1; }     /* external wrenches: generic kernels only */
  static RKFD_HD int rk_slot(const ModelDev &){ return RK; }
  static RKFD_HD int nq(const ModelDev &){ return NL_ - 1; }
  static RKFD_HD int sc(int i, const LinkDev &){ return RG_ ? PER*i + 9 : 4*(i-1); }
};
inline bool spec_serial_rev_rolled_match(const ModelDev &m, int NL, int RG = 0, int GEN = 0){
  if( m.nfw > 1 || m.npair > m.npair_static || m.nslide > 0 || m.nfext > 0 ) return false;   /* slide mode, external wrenches: generic kernel only */
  if( RG ? !( m.has_rigid && m.nrg == 1 && m.rigid_link == NL-1 ) : m.has_rigid ) return false;
  if( m.nl != NL || NL < 2 ) return false;
  for(int i=0;i<NL;i++){
    const LinkDev &L = m.link[i];
    if( i == 0 ){ if( L.parent >= 0 || L.jtype != J_FIXED || L.cell_end > L.cell_begin ) return false; continue; }
    if( L.jtype != J_REVOL || L.parent != i-1 || !L.serial || L.qofs != i-1 ) return false;
    if( !GEN && L.rcls != RO_RXP && L.rcls != RO_RXM ) return false;
    if( i != NL-1 && L.cell_end > L.cell_begin ) return false;
  }
  return true;
}

/* does the flattened model have the shape SpecSerialRev<.,NL,CLS> assumes? (host side) */
inline bool spec_serial_rev_match(const ModelDev &m, int NL, unsigned CLS){
  if( m.has_rigid || m.nl != NL || NL < 2 || m.nfw > 1 || m.npair > m.npair_static || m.nslide > 0 || m.nfext > 0 ) return false;
  for(int i=0;i<NL;i++){
    const LinkDev &L = m.link[i];
    if( i == 0 ){ if( L.parent >= 0 || L.jtype != J_FIXED || L.cell_end > L.cell_begin ) return false; continue; }
    if( L.jtype != J_REVOL || L.parent != i-1 || !L.serial || L.qofs != i-1 ) return false;
    if( L.rcls == RO_GENERAL || L.rcls != (int)((CLS >> (2*(i-1))) & 3u) ) return false;
    if( i != NL-1 && L.cell_end > L.cell_begin ) return false;
  }
  return true;
}

/* compiled specialisations: (id, links, rotation classes).  1: the 7-DoF arm of BASELINE.json (fixed base + 7
 * revolute links, frames alternating Rx(-90)/Rx(+90)); 2: fixed base + 2 parallel revolute links (arm_2DoF.ztk) */
#define RKFD_SPEC_TABLE(X) X(3, 8, 0x3BBBu, 1) X(4, 3, 0x5u, 1) X(1, 8, 0x3BBBu, 0) X(2, 3, 0x5u, 0)
/* rolled specialisations: (id, links, rigid layout, general frames); 5/6: fixed base + 7/6 revolute links with
 * quarter-turn frames, 7: the same with rigid pairs on the last link, 8-10: general frames, 2/6/7 revolute links */
#define RKFD_SPEC_ROLLED_TABLE(X) X(5, 8, 0, 0) X(6, 7, 0, 0) X(7, 8, 1, 0) X(8, 3, 0, 1) X(9, 7, 0, 1) X(10, 8, 0, 1)
template <int ID> struct SpecOf { using type = SpecGeneric; };
template <> struct SpecOf<11> { using type = SpecGenericTM; };
#define RKFD_SPEC_X(id, nl, cls, tm) template <> struct SpecOf<id> { using type = SpecSerialRev<id, nl, cls, tm>; };
RKFD_SPEC_TABLE(RKFD_SPEC_X)
#undef RKFD_SPEC_X
#define RKFD_SPEC_X(id, nl, rg, gen) template <> struct SpecOf<id> { using type = SpecSerialRevRolled<id, nl, rg, gen>; };
RKFD_SPEC_ROLLED_TABLE(RKFD_SPEC_X)
#undef RKFD_SPEC_X
/* specialisation ids the model is eligible for (bit id set; 0: generic kernel only), and their scratch sizes */
inline unsigned spec_match_mask(const ModelDev &m){
  unsigned mask = 0;
#define RKFD_SPEC_X(id, nl, cls, tm) if( spec_serial_rev_match(m, nl, cls) ) mask |= 1u << id;
  RKFD_SPEC_TABLE(RKFD_SPEC_X)
#undef RKFD_SPEC_X
#define RKFD_SPEC_X(id, nl, rg, gen) if( spec_serial_rev_rolled_match(m, nl, rg, gen) ) mask |= 1u << id;
  RKFD_SPEC_ROLLED_TABLE(RKFD_SPEC_X)
#undef RKFD_SPEC_X
  return mask;
}
inline int spec_match_rolled(const ModelDev &m){
#define RKFD_SPEC_X(id, nl, rg, gen) if( spec_serial_rev_rolled_match(m, nl, rg, gen) ) return id;
  RKFD_SPEC_ROLLED_TABLE(RKFD_SPEC_X)
#undef RKFD_SPEC_X
  return 0;
}
inline int spec_match(const ModelDev &m, int want_tm = 1){     /* preferred id: first in table order with tm == want_tm */
#define RKFD_SPEC_X(id, nl, cls, tm) if( tm == want_tm && spec_serial_rev_match(m, nl, cls) ) return id;
  RKFD_SPEC_TABLE(RKFD_SPEC_X)
#undef RKFD_SPEC_X
  return 0;
}
inline int spec_nscratch(int id){
#define RKFD_SPEC_X(sid, nl, cls, tm) if( id == sid ) return SpecSerialRev<sid, nl, cls, tm>::NSCRATCH;
  RKFD_SPEC_TABLE(RKFD_SPEC_X)
#undef RKFD_SPEC_X
#define RKFD_SPEC_X(sid, nl, rg, gen) if( id == sid ) return SpecSerialRevRolled<sid, nl, rg, gen>::NSCRATCH;
  RKFD_SPEC_ROLLED_TABLE(RKFD_SPEC_X)
#undef RKFD_SPEC_X
  return 0;
}
inline int spec_ntspace(int id){
  if( id == SPEC_GENERIC_TM ) return SPEC_GENERIC_TM_MAX_T;
#define RKFD_SPEC_X(sid, nl, cls, tm) if( id == sid ) return SpecSerialRev<sid, nl, cls, tm>::NTSPACE;
  RKFD_SPEC_TABLE(RKFD_SPEC_X)
#undef RKFD_SPEC_X
#define RKFD_SPEC_X(sid, nl, rg, gen) if( id == sid ) return SpecSerialRevRolled<sid, nl, rg, gen>::NTSPACE;
  RKFD_SPEC_ROLLED_TABLE(RKFD_SPEC_X)
#undef RKFD_SPEC_X
  return 0;
}

/* explicit Runge-Kutta coefficients times dt ([EXT A-9]; zODE2AssignRegular menu) */
inline ModelDev::RK rk_coef(double dt, int integrator){
  const double r2 = sqrt(2.0); ModelDev::RK k;
  k.c21 = 0.5*dt; k.c31 = ((r2-1.0)/2.0)*dt; k.c32 = (1.0-1.0/r2)*dt; k.c42 = (-1.0/r2)*dt; k.c43 = (1.0+1.0/r2)*dt;
  k.b1 = (1.0/6.0)*dt; k.b2 = ((2.0-r2)/6.0)*dt; k.b3 = ((2.0+r2)/6.0)*dt; k.b4 = (1.0/6.0)*dt; k.ns = 4;
  if( integrator == 1 ){ k.c31 = 0.0; k.c32 = 0.5*dt; k.c42 = 0.0; k.c43 = dt; k.b2 = (2.0/6.0)*dt; k.b3 = (2.0/6.0)*dt; }
  else if( integrator == 2 ){ k.ns = 1; k.b1 = dt; }
  else if( integrator == 3 ){ k.ns = 2; k.c21 = dt; k.b1 = 0.5*dt; k.b4 = 0.5*dt; }
  return k;
}

template <class Ctx, class Spec = SpecGeneric>
struct Core {
  Ctx &c;
  unsigned int piv;             /* joint friction pivot: bit j = dof j kinetic */
  unsigned long long cfl;       /* contact flags, the word `cw` of them: bit 2f active, bit 2f+1 kinetic */
  int cw;
  int bad;
  unsigned wk = 0;              /* work class of the last rigid solve (StateDev::work) */
  int rk0;                      /* first slot of the integrator stage state (QS, QDS, PQ, PQD) */
  /* committed state (buffer `cur` of StateDev::q/qd) and the output buffer, where the running combination of a step becomes
   * the next committed state; selected once, swapped when a step commits.  Indexing StateDev::q with the run-time `cur` at
   * every access instead makes nvcc keep a copy of the whole StateDev on the stack and reload the pointers from there. */
  double *qc, *qdc, *qn, *qdn;

  RKFD_HD explicit Core(Ctx &ctx) : c(ctx), piv(0), cfl(0), cw(0), bad(0), rk0(0),
    qc(ctx.cur ? ctx.st.q[1] : ctx.st.q[0]), qdc(ctx.cur ? ctx.st.qd[1] : ctx.st.qd[0]),
    qn(ctx.cur ? ctx.st.q[0] : ctx.st.q[1]), qdn(ctx.cur ? ctx.st.qd[0] : ctx.st.qd[1]) {}
  RKFD_HD void commit_swap(){ double *t = qc; qc = qn; qn = t; t = qdc; qdc = qdn; qdn = t; }

  /* the flag word the following code works on (warp-uniform: decided by the model) */
  RKFD_HD void flag_select(int w){
    if( Spec::NL != 0 ) return;      /* the arm specialisations only match single-word worlds (spec_*_match) */
    if( w != cw ){ c.st.cflags[(size_t)cw*c.st.ld + c.e] = cfl; cfl = c.st.cflags[(size_t)w*c.st.ld + c.e]; cw = w; }
  }

  /* link properties: the compile-time tag when it knows, the Spec accessor (table / unrolled index) otherwise */
  template <class Kt> static RKFD_HD int JT(int i, const LinkDev &L){ return Kt::jt >= 0 ? Kt::jt : Spec::jtype(i,L); }
  template <class Kt> static RKFD_HD int CLS(int i, const LinkDev &L){ return Kt::cls >= 0 ? Kt::cls : Spec::rcls(i,L); }
  template <class Kt> static RKFD_HD bool ROOT(int i, const LinkDev &L){ return Kt::root >= 0 ? Kt::root != 0 : Spec::parent(i,L) < 0; }
  template <class Kt> static RKFD_HD bool SER(int i, const LinkDev &L){ return Kt::root >= 0 ? Kt::root == 0 : Spec::serial(i,L) != 0; }
  /* link loops: base -> tip and tip -> base.  f(i, tag) is the pass body */
  template <class F> RKFD_HD void links_fwd(const ModelDev &m, F &&f){
    if constexpr ( Spec::ROLL != 0 ){
      f(0, LinkTag<J_FIXED, RO_GENERAL, 1>{});
#pragma unroll (ROLL_UNROLL)
      for(int i=1;i<Spec::NL;i++) f(i, LinkTag<J_REVOL, Spec::RCLS, 0>{});
    } else {
      const int NLc = Spec::nl(m);
#pragma unroll (Spec::UNROLL)
      for(int i=0;i<NLc;i++) f(i, TagRT{});
    }
  }
  template <class F> RKFD_HD void links_bwd(const ModelDev &m, F &&f){
    if constexpr ( Spec::ROLL != 0 ){
#pragma unroll (ROLL_UNROLL)
      for(int i=Spec::NL-1;i>=1;i--) f(i, LinkTag<J_REVOL, Spec::RCLS, 0>{});
      f(0, LinkTag<J_FIXED, RO_GENERAL, 1>{});
    } else {
      const int NLc = Spec::nl(m);
#pragma unroll (Spec::UNROLL)
      for(int i=NLc-1;i>=0;i--) f(i, TagRT{});
    }
  }

  /* T space: integrator stage state and per-joint (sin, cos, 1/D, u) - tensor memory in the TM specialisations,
   * the scratch column otherwise */
  RKFD_HD double T(int k){ return c.TL(k); }
  RKFD_HD void Tw(int k, double v){ c.TS(k, v); }
  /* per-joint (sin, cos, 1/D, u): T space, or the scratch column when the specialisation says so (Spec::SCS) */
  RKFD_HD double Q(int k){ return Spec::SCS ? c.S(k) : c.TL(k); }
  RKFD_HD void Qw(int k, double v){ if( Spec::SCS ) c.S(k) = v; else c.TS(k, v); }
  RKFD_HD void Q2(int k, double &a, double &b){ if( Spec::SCS ){ a = c.S(k); b = c.S(k+1); } else c.TL2(k, a, b); }
  RKFD_HD V3 t3(int k){ const double x = c.TL(k), y = c.TL(k+1), z = c.TL(k+2); return v3(x, y, z); }   /* k is arbitrary: no paired (x4) load */
  RKFD_HD void tw3(int k, V3 v){ c.TS(k, v.x); c.TS(k+1, v.y); c.TS(k+2, v.z); }
  RKFD_HD V3 ld3(int k){ return v3(c.S(k), c.S(k+1), c.S(k+2)); }
  RKFD_HD void st3(int k, V3 v){ c.S(k)=v.x; c.S(k+1)=v.y; c.S(k+2)=v.z; }
  RKFD_HD M3 ldm(int k){ M3 m; m.xx=c.S(k); m.xy=c.S(k+1); m.xz=c.S(k+2); m.yx=c.S(k+3); m.yy=c.S(k+4); m.yz=c.S(k+5); m.zx=c.S(k+6); m.zy=c.S(k+7); m.zz=c.S(k+8); return m; }
  RKFD_HD void stm(int k, const M3 &m){ c.S(k)=m.xx; c.S(k+1)=m.xy; c.S(k+2)=m.xz; c.S(k+3)=m.yx; c.S(k+4)=m.yy; c.S(k+5)=m.yz; c.S(k+6)=m.zx; c.S(k+7)=m.zy; c.S(k+8)=m.zz; }
  RKFD_HD S3 lds(int k){ S3 s; s.xx=c.S(k); s.xy=c.S(k+1); s.xz=c.S(k+2); s.yy=c.S(k+3); s.yz=c.S(k+4); s.zz=c.S(k+5); return s; }

  static RKFD_HD M3 org_R(const LinkDev &L){ M3 m; m.xx=L.Ro[0]; m.xy=L.Ro[1]; m.xz=L.Ro[2]; m.yx=L.Ro[3]; m.yy=L.Ro[4]; m.yz=L.Ro[5]; m.zx=L.Ro[6]; m.zy=L.Ro[7]; m.zz=L.Ro[8]; return m; }
  static RKFD_HD V3 org_p(const LinkDev &L){ return v3(L.po[0],L.po[1],L.po[2]); }

  /* link frame w.r.t. parent and joint velocity (vJ,wJ, link frame) from the stage state and the joint data
   * cached by pass 1 ([EXT A-3]) */
  /* VEL = false: the transform only (the contact-solve probes: no T-space access, which must be warp-uniform) */
  template <class Kt, bool VEL = true>
  RKFD_HD XF joint_xform(const ModelDev &m, const LinkDev &L, int i, V3 &vJ, V3 &wJ){
    const int sl = Spec::slot(i,L), qs = rk0 + Spec::qofs(i,L), qds = rk0 + Spec::nq(m) + Spec::qofs(i,L);
    XF x; x.fast = 0; x.cls = CLS<Kt>(i,L); x.sg = ro_sign(x.cls, L.rsg); x.c = 1.0; x.s = 0.0;
    x.pz = L.pz;      /* revolute / fixed joint with org position (0, 0, z): decided once on the host (rkfd_model.cpp) */
    vJ = v3(0,0,0); wJ = v3(0,0,0);
    switch(JT<Kt>(i,L)){
    case J_REVOL: {
      Q2(Spec::sc(i,L), x.s, x.c); x.p = org_p(L);
      if( CLS<Kt>(i,L) != RO_GENERAL ){ x.fast = 1; x.ptl = rz_tmul(x.c, x.s, v3(L.pol[0],L.pol[1],L.pol[2])); }
      else {
        const M3 Ro = org_R(L); const V3 o0 = col0(Ro), o1 = col1(Ro);
        x.R = from_cols(x.c*o0 + x.s*o1, x.c*o1 - x.s*o0, col2(Ro)); x.ptl = tmul(x.R, x.p);
      }
      if( VEL ) wJ.z = T(qds);
    } break;
    case J_PRISM: {
      x.R = org_R(L); x.p = org_p(L) + T(qs)*col2(x.R); x.ptl = tmul(x.R, x.p); if( VEL ) vJ.z = T(qds);
    } break;
    case J_SPHER: {
      x.R = ldm(sl+27); x.p = org_p(L); x.ptl = tmul(x.R, x.p);
      if( VEL ) wJ = tmul(x.R, mul(org_R(L), t3(qds)));
    } break;
    case J_FLOAT: {
      x.R = ldm(sl+6); x.p = ld3(sl+15); x.ptl = tmul(x.R, x.p);
      const M3 Ro = org_R(L);
      if( VEL ){ vJ = tmul(x.R, mul(Ro, t3(qds))); wJ = tmul(x.R, mul(Ro, t3(qds+3))); }
    } break;
    case J_BRFLOAT: {      /* frame as for the float joint; joint velocities only once it has broken (flag cached in the column by pass 1) */
      x.R = ldm(sl+6); x.p = ld3(sl+15); x.ptl = tmul(x.R, x.p);
      if( VEL ){ const M3 Ro = org_R(L); const V3 v = t3(qds), w = t3(qds+3);
        if( c.S(sl+45) != 0.0 ){ vJ = tmul(x.R, mul(Ro, v)); wJ = tmul(x.R, mul(Ro, w)); } }
    } break;
    case J_CYLIN: case J_HOOKE: {
      x.R = ldm(sl+17); x.p = ld3(sl+26); x.ptl = tmul(x.R, x.p);
      if( VEL ){ const double v0 = T(qds), v1 = T(qds+1);
        if( JT<Kt>(i,L) == J_CYLIN ){ vJ.z = v0; wJ.z = v1; }
        else { const double s1 = c.S(sl+29), c1 = c.S(sl+30); wJ = v3(-s1*v0, v1, c1*v0); } }
    } break;
    default: x.R = org_R(L); x.p = org_p(L); x.ptl = v3(L.pol[0],L.pol[1],L.pol[2]); break;
    }
    return x;
  }
  /* the joint type the ABA passes see: a breakable float is a fixed joint until it breaks, a float joint afterwards */
  RKFD_HD int eff_jt(int jt, int sl){ return jt == J_BRFLOAT ? ( c.S(sl+45) != 0.0 ? (int)J_FLOAT : (int)J_FIXED ) : jt; }
  /* free 6-DoF joint, inward pass: a0 = -IA^-1 pA into the column (and IA^-1 for the contact-solve probes) */
  RKFD_HD void float_project(const S3 &A, const M3 &B, const S3 &C, V3 pf, V3 pn, int sl, bool keep_inverse){
    double a[36];
    a[0]=A.xx; a[1]=A.xy; a[2]=A.xz; a[6]=A.xy; a[7]=A.yy; a[8]=A.yz; a[12]=A.xz; a[13]=A.yz; a[14]=A.zz;
    a[3]=B.xx; a[4]=B.xy; a[5]=B.xz; a[9]=B.yx; a[10]=B.yy; a[11]=B.yz; a[15]=B.zx; a[16]=B.zy; a[17]=B.zz;
    a[18]=B.xx; a[19]=B.yx; a[20]=B.zx; a[24]=B.xy; a[25]=B.yy; a[26]=B.zy; a[30]=B.xz; a[31]=B.yz; a[32]=B.zz;
    a[21]=C.xx; a[22]=C.xy; a[23]=C.xz; a[27]=C.xy; a[28]=C.yy; a[29]=C.yz; a[33]=C.xz; a[34]=C.yz; a[35]=C.zz;
    spd6_inverse(a);
    const double b[6] = {pf.x,pf.y,pf.z,pn.x,pn.y,pn.z};
#pragma unroll
    for(int r=0;r<6;r++){ double t = 0;
#pragma unroll
      for(int k=0;k<6;k++) t -= a[6*r+k]*b[k];
      c.S(sl+r) = t; }
    if( keep_inverse ){ int k = 0;
#pragma unroll
      for(int r=0;r<6;r++)
#pragma unroll
        for(int q=0;q<6;q++) if(q>=r){ c.S(sl+18+k) = a[6*r+q]; k++; } }
  }
  /* motion axes of the 2-DoF joints in the link frame ([EXT] cylindrical: (z; 0), (0; z); hooke: (0; Ry(q1)^T z), (0; y)) */
  RKFD_HD void axes2(int jt, int sl, V3 &l0, V3 &a0, V3 &l1, V3 &a1){
    if( jt == J_CYLIN ){ l0 = v3(0,0,1); a0 = v3(0,0,0); l1 = v3(0,0,0); a1 = v3(0,0,1); }
    else { l0 = v3(0,0,0); a0 = v3(-c.S(sl+29), 0.0, c.S(sl+30)); l1 = v3(0,0,0); a1 = v3(0,1,0); }
  }
  /* bias-force change (dpf, dpn) at a 2-DoF joint: stores du = -S^T dp, returns the change handed to the parent side */
  RKFD_HD void probe2_in(int jt, int sl, V3 dpf, V3 dpn, double (&du)[2], V3 &paf, V3 &pan){
    V3 l0, a0, l1, a1; axes2(jt, sl, l0, a0, l1, a1);
    du[0] = -(dot(l0,dpf) + dot(a0,dpn)); du[1] = -(dot(l1,dpf) + dot(a1,dpn));
    const double k0 = c.S(sl+12)*du[0] + c.S(sl+13)*du[1], k1 = c.S(sl+13)*du[0] + c.S(sl+14)*du[1];
    paf = dpf + k0*ld3(sl) + k1*ld3(sl+6); pan = dpn + k0*ld3(sl+3) + k1*ld3(sl+9);
  }
  /* acceleration response of a 2-DoF joint to du with the transformed parent acceleration (xl, xa) */
  RKFD_HD void probe2_out(int jt, int sl, const double (&du)[2], V3 &xl, V3 &xa){
    V3 l0, a0, l1, a1; axes2(jt, sl, l0, a0, l1, a1);
    const double r0 = du[0] - (dot(ld3(sl),xl) + dot(ld3(sl+3),xa)), r1 = du[1] - (dot(ld3(sl+6),xl) + dot(ld3(sl+9),xa));
    const double q0 = c.S(sl+12)*r0 + c.S(sl+13)*r1, q1 = c.S(sl+13)*r0 + c.S(sl+14)*r1;
    xl = xl + q0*l0 + q1*l1; xa = xa + q0*a0 + q1*a1;
  }

  /* [EXT A-10] closest face of the box for a vertex inside it: first minimum depth over x,y,z; outward normal,
   * right-handed tangents, projection of the vertex on that face (box frame) */
  static RKFD_HD void box_face(const BoxDev &bx, const M3 &Rb, V3 vb, double dx, double dy, double dz,
                               V3 &n, V3 &t1, V3 &t2, V3 &prob){
    int amin = 0; double dmin = dx;
    if( dy < dmin ){ dmin = dy; amin = 1; }
    if( dz < dmin ){ dmin = dz; amin = 2; }
    const double vba = amin==0 ? vb.x : ( amin==1 ? vb.y : vb.z );
    const double sg = vba >= 0 ? 1.0 : -1.0;
    const V3 b0 = col0(Rb), b1 = col1(Rb), b2 = col2(Rb);
    n  = sg*( amin==0 ? b0 : ( amin==1 ? b1 : b2 ) );
    t1 =      amin==0 ? b1 : ( amin==1 ? b2 : b0 );
    t2 = sg*( amin==0 ? b2 : ( amin==1 ? b0 : b1 ) );
    prob = vb;
    if( amin==0 ) prob.x = sg*bx.half[0]; else if( amin==1 ) prob.y = sg*bx.half[1]; else prob.z = sg*bx.half[2];
  }
  static RKFD_HD M3 box_R(const BoxDev &bx){ M3 Rb; Rb.xx=bx.R[0]; Rb.xy=bx.R[1]; Rb.xz=bx.R[2]; Rb.yx=bx.R[3]; Rb.yy=bx.R[4]; Rb.yz=bx.R[5]; Rb.zx=bx.R[6]; Rb.zy=bx.R[7]; Rb.zz=bx.R[8]; return Rb; }

  /* does pair pr involve a cell in slide mode?  Always false in the model specialisations (they do not match such worlds): their
   * kernels carry none of the slide code */
  static RKFD_HD bool has_slide(const PairDev &pr){ if constexpr ( Spec::NL != 0 ) return false; else return (pr.slinfo & 0xffff) != 0; }
  /* ---- slide mode of collision cells ("fake crawler": rkFDLinkAddSlideVel rkfd_util.c:26-40, rkFDUpdateRefSlide :218-237).
   * Belt direction of slide entry sd, carried by the frame (R, pw), at world point p: (R axis) x (p - pw) without its normal
   * component; returns its norm */
  static RKFD_HD double slide_dir(const SlideDev &sd, const M3 &R, V3 pw, V3 p, V3 n, V3 &sv){
    sv = cross(mul(R, v3(sd.axis[0], sd.axis[1], sd.axis[2])), p - pw); sv = sv + (-dot(sv, n))*n; return norm(sv); }
  static RKFD_HD M3 slide_lR(const SlideDev &sd){ M3 r; r.xx=sd.lR[0]; r.xy=sd.lR[1]; r.xz=sd.lR[2]; r.yx=sd.lR[3]; r.yy=sd.lR[4]; r.yz=sd.lR[5]; r.zx=sd.lR[6]; r.zy=sd.lR[7]; r.zz=sd.lR[8]; return r; }
  /* what the belts add to the relative velocity (vertex's cell minus partner) of pair pr at world point p with contact normal n;
   * (Rv, pv): frame of the vertex's link; (Rp, pp): frame of a MOVING partner link (a static partner's frame is in its entry) */
  static RKFD_HD V3 slide_vel(const ModelDev &m, const PairDev &pr, const M3 &Rv, V3 pv, const M3 &Rp, V3 pp, V3 p, V3 n){
    V3 out = v3(0,0,0); const int sc = (pr.slinfo & 255) - 1, sb = ((pr.slinfo >> 8) & 255) - 1;
    if( sc >= 0 ){ V3 sv; const double nv = slide_dir(m.slide[sc], Rv, pv, p, n, sv); if( !(fabs(nv) < ZTOL) ) out = out + (m.slide[sc].vel/nv)*sv; }
    if( sb >= 0 ){ const SlideDev &sd = m.slide[sb]; V3 sv; const bool mov = pr.mbox >= 0;
      const double nv = slide_dir(sd, mov ? Rp : slide_lR(sd), mov ? pp : v3(sd.lp[0], sd.lp[1], sd.lp[2]), p, n, sv);
      if( !(fabs(nv) < ZTOL) ) out = out + (-sd.vel/nv)*sv; }
    return out; }
  /* the anchor of a sticking contact rides on the belt: shift of the anchor in the BOX frame (Rbw = world rotation of the box,
   * Rpl = world rotation of the partner's link).  The reference adds R_k^T sv to _ref with k = pd->cell[1]'s link when the
   * sliding cell is the vertex's cell, else pd->cell[0]'s link, and _ref lives in the partner's frame: world shift
   * R_partner R_k^T sv (= sv whenever the sliding cell is pd->cell[0]) - mirrored */
  static RKFD_HD V3 slide_ref_shift(const ModelDev &m, const PairDev &pr, const M3 &Rv, V3 pv, const M3 &Rpl, V3 pp, const M3 &Rbw, V3 p, V3 n){
    V3 db = v3(0,0,0); const int sc = (pr.slinfo & 255) - 1, sb = ((pr.slinfo >> 8) & 255) - 1;
    const bool vfirst = (pr.slinfo >> 16) & 1, mov = pr.mbox >= 0;
    for(int i=0;i<2;i++){
      const bool is_v = vfirst ? i == 0 : i == 1; const int idx = is_v ? sc : sb;
      if( idx < 0 ) continue;
      const SlideDev &sd = m.slide[idx]; V3 sv;
      const double nv = is_v ? slide_dir(sd, Rv, pv, p, n, sv) : slide_dir(sd, mov ? Rpl : slide_lR(sd), mov ? pp : v3(sd.lp[0], sd.lp[1], sd.lp[2]), p, n, sv);
      if( fabs(nv) < ZTOL ) continue;
      const double k = ( is_v ? -1.0 : 1.0 )*m.dt*sd.vel/nv;
      sv = k*sv;
      const bool k_is_v = is_v ? !vfirst : vfirst;
      const V3 dw = mul(Rpl, k_is_v ? tmul(Rv, sv) : tmul(Rpl, sv));
      db = db + tmul(Rbw, dw);
    }
    return db; }
  static RKFD_HD M3 box_lR(const BoxDev &bx){ M3 r; r.xx=bx.lR[0]; r.xy=bx.lR[1]; r.xz=bx.lR[2]; r.yx=bx.lR[3]; r.yy=bx.lR[4]; r.yz=bx.lR[5]; r.zx=bx.lR[6]; r.zy=bx.lR[7]; r.zz=bx.lR[8]; return r; }

  /* ---- contact of the cells carried by link i: vertex-in-box detection ([EXT A-10]), elastic pairs:
   * penalty force + Coulomb clamp + wrench accumulation (rkfd_penalty.c:11-31, rkfd_util.c:239-282).
   * Two phases per (cell, box) pair so that a warp does not walk through the expensive force code once per
   * candidate vertex: (A) the cheap inside test of every vertex, all lanes in lockstep, gives each lane the bit
   * mask of its vertices in contact; (B) every lane then serves its own vertices in ascending order - the warp
   * iterates max-over-lanes(#contacts) times (typically 1-4) instead of #vertices (8) times.  The order of the
   * wrench summation per environment is unchanged (pair, vertex). */
  RKFD_HD V6 contacts(const ModelDev &m, const LinkDev &L, const M3 &Rw, V3 pw, V3 vl, V3 om, bool ref){
    V6 w; w.l = v3(0,0,0); w.a = v3(0,0,0);
    const V3 vlw = mul(Rw, vl), omw = mul(Rw, om);     /* rkFDLinkPointWldVel (rkfd_util.c:14-24): world velocity of the link origin, world angular velocity */
    for(int ci=L.cell_begin; ci<L.cell_end; ci++){
      const CellDev &cl = m.cell[ci];
      for(int pi=cl.pair_begin; pi<cl.pair_end; pi++){
        const PairDev &pr = m.pair[pi]; const BoxDev &bx = m.box[pr.box];
        const M3 Rb = box_R(bx);
        const V3 pb = v3(bx.p[0],bx.p[1],bx.p[2]);
        /* (A) detection: vertex in the box frame = Rb^T (pw - pb) + (Rb^T Rw) vloc, the two factors once per pair */
        const M3 Mb = tmm(Rb, Rw); const V3 ob = tmul(Rb, pw - pb);
        /* chunks of 32 vertices: one flag word each */
        /* (the arm specialisations only match single-word worlds: one chunk, flag position = slot) */
        const int c0end = Spec::NL != 0 ? 1 : cl.nvert;
        for(int c0_=0; c0_<c0end; c0_+=32){
        const int c0 = Spec::NL != 0 ? 0 : c0_;
        const int nvc = Spec::NL != 0 ? cl.nvert : ( cl.nvert - c0 < 32 ? cl.nvert - c0 : 32 );
        const int sh = Spec::NL != 0 ? pr.sofs : ( (pr.fofs + c0) & 31 );
        flag_select((pr.fofs + c0) >> 5);
        unsigned in = 0;
        for(int k=0;k<nvc;k++){
          const int s = pr.sofs + c0 + k, vi = cl.vofs + c0 + k;
          const V3 vloc = v3(m.vert[3*vi], m.vert[3*vi+1], m.vert[3*vi+2]);
          const V3 vb = ob + mul(Mb, vloc);
          const double dx = bx.half[0]-fabs(vb.x), dy = bx.half[1]-fabs(vb.y), dz = bx.half[2]-fabs(vb.z);
          const bool inside = (dx > -ZTOL) && (dy > -ZTOL) && (dz > -ZTOL);
          if( inside ) in |= 1u << k;
          else { cfl &= ~(3ull << (2*(sh+k))); if( ref ){ c.gst(c.st.cf, 3*s, 0.0); c.gst(c.st.cf, 3*s+1, 0.0); c.gst(c.st.cf, 3*s+2, 0.0); } }
        }
        /* (B) the lane's own contacts */
        while( c.any(in != 0) ){
          if( in == 0 ) continue;
          const int k = RKFD_FFS32(in) - 1; in &= in - 1;
          const int s = pr.sofs + c0 + k, vi = cl.vofs + c0 + k;
          const unsigned long long abit = 1ull << (2*(sh+k)), kbit = 2ull << (2*(sh+k));
          const V3 vloc = v3(m.vert[3*vi], m.vert[3*vi+1], m.vert[3*vi+2]);
          const V3 vw = pw + mul(Rw, vloc);
          const V3 vb = tmul(Rb, vw - pb);
          const double dx = bx.half[0]-fabs(vb.x), dy = bx.half[1]-fabs(vb.y), dz = bx.half[2]-fabs(vb.z);
          V3 n, t1, t2, prob;
          box_face(bx, Rb, vb, dx, dy, dz, n, t1, t2, prob);
          V3 refb;
          if( !(cfl & abit) ){           /* new contact: {SF, _ref = _pro} */
            cfl = (cfl | abit) & ~kbit; refb = prob;
            c.gst(c.st.cref, 3*s, refb.x); c.gst(c.st.cref, 3*s+1, refb.y); c.gst(c.st.cref, 3*s+2, refb.z);
          } else refb = v3(c.gld(c.st.cref,3*s), c.gld(c.st.cref,3*s+1), c.gld(c.st.cref,3*s+2));
          if( pr.type != C_ELASTIC ) continue;     /* rigid pairs are solved by the rigid path */
          const V3 refw = pb + mul(Rb, refb);
          const V3 d = vw - refw;
          /* rkFDLinkPointWldVel (rkfd_util.c:14-24); the static partner contributes 0 */
          V3 vr = vlw + cross(omw, vw - pw);
          if( has_slide(pr) ) vr = vr + slide_vel(m, pr, Rw, pw, Rw, pw, vw, n);
          V3 f = (-pr.E)*d + (-1.0*(pr.V + pr.E*m.dt))*vr;
          if( dot(f,n) < 0.0 ){ if( ref ){ c.gst(c.st.cf,3*s,f.x); c.gst(c.st.cf,3*s+1,f.y); c.gst(c.st.cf,3*s+2,f.z); } continue; }
          /* rkFDContactForceModifyFriction */
          const double fn = dot(f,n), f1 = dot(f,t1), f2 = dot(f,t2);
          const double fs = sqrt(f1*f1 + f2*f2);
          const double mu = (cfl & kbit) ? pr.KF : pr.SF;
          if( !(fabs(fs) < ZTOL) && fs > mu*fn ){
            V3 v = vr + (-dot(vr,n))*n;
            const double vs = norm(v);
            f = fn*n;
            if( !(fabs(vs) < ZTOL) ){
              f = f + ((-(1.0 - exp(-1.0*m.friction_weight*vs))*pr.KF*fn)/vs)*v;
            }
            if( ref ){ cfl |= kbit; c.gst(c.st.cref,3*s,prob.x); c.gst(c.st.cref,3*s+1,prob.y); c.gst(c.st.cref,3*s+2,prob.z); }
          } else if( ref ){
            cfl &= ~kbit;
            if( has_slide(pr) ){ const V3 nr = refb + slide_ref_shift(m, pr, Rw, pw, box_lR(bx), v3(0,0,0), Rb, vw, n);
              c.gst(c.st.cref,3*s,nr.x); c.gst(c.st.cref,3*s+1,nr.y); c.gst(c.st.cref,3*s+2,nr.z); }
          }
          /* rkFDContactForcePushWrench: (f, pos x f) at the link origin, link axes */
          const V3 pos = tmul(Rw, vw - pw);
          const V3 fl = tmul(Rw, f);
          w.l = w.l + fl; w.a = w.a + cross(pos, fl);
          if( ref ){ c.gst(c.st.cf,3*s,f.x); c.gst(c.st.cf,3*s+1,f.y); c.gst(c.st.cf,3*s+2,f.z); }
        }
        }
      }
    }
    return w;
  }

  /* ---- contacts between two MOVING links ([EXT A-10] extended: the vertices of a cell against a box primitive carried by
   * another link; reference: rkFDChainPointRelativeVel rkfd_util.c:42-60 - the velocity of the vertex's link minus the box
   * link's at the contact point - and rkFDContactForcePushWrench rkfd_util.c:268-282 - the force on the vertex's link, its
   * opposite on the partner, both at the contact point).  Runs after pass 1, when every link frame of the evaluation is known
   * (frame slots of the links involved).  Elastic pairs: rkFDSolverPenalty (rkfd_penalty.c:11-31); rigid pairs: detection and
   * the persistent vertex state only, their forces come from the dense rigid path (rigid_solve).  Generic kernel only. */
  RKFD_HD void contacts_moving(const ModelDev &m, bool ref){
    for(int pi=m.npair_static; pi<m.npair; pi++){
      const PairDev &pr = m.pair[pi]; const CellDev &cl = m.cell[pr.cell]; const MBoxDev &mb = m.mbox[pr.mbox];
      const LinkDev &LA = m.link[cl.link], &LB = m.link[mb.link];
      const int fa = Spec::frame_slot(cl.link, LA), fb = Spec::frame_slot(mb.link, LB), wa = Spec::wext_slot(cl.link, LA), wb = Spec::wext_slot(mb.link, LB);
      const M3 Rw = ldm(fa); const V3 pw = ld3(fa+9);
      const M3 RwB = ldm(fb); const V3 pwB = ld3(fb+9);
      M3 Rl; Rl.xx=mb.R[0]; Rl.xy=mb.R[1]; Rl.xz=mb.R[2]; Rl.yx=mb.R[3]; Rl.yy=mb.R[4]; Rl.yz=mb.R[5]; Rl.zx=mb.R[6]; Rl.zy=mb.R[7]; Rl.zz=mb.R[8];
      const M3 Rb = mm(RwB, Rl); const V3 pb = pwB + mul(RwB, v3(mb.p[0], mb.p[1], mb.p[2]));
      BoxDev bx; for(int i=0;i<3;i++) bx.half[i] = mb.half[i];
      const V3 vlw = mul(Rw, ld3(fa+12)), omw = mul(Rw, ld3(fa+15)), vlwB = mul(RwB, ld3(fb+12)), omwB = mul(RwB, ld3(fb+15));
      V6 wA, wB; wA.l = wA.a = wB.l = wB.a = v3(0,0,0);
      for(int c0=0; c0<cl.nvert; c0+=32){
        const int nvc = cl.nvert - c0 < 32 ? cl.nvert - c0 : 32, sh = (pr.fofs + c0) & 31;
        flag_select((pr.fofs + c0) >> 5);
        unsigned in = 0;
        for(int k=0;k<nvc;k++){
          const int s = pr.sofs + c0 + k, vi = cl.vofs + c0 + k;
          const V3 vb = tmul(Rb, pw + mul(Rw, v3(m.vert[3*vi], m.vert[3*vi+1], m.vert[3*vi+2])) - pb);
          const bool inside = (bx.half[0]-fabs(vb.x) > -ZTOL) && (bx.half[1]-fabs(vb.y) > -ZTOL) && (bx.half[2]-fabs(vb.z) > -ZTOL);
          if( inside ) in |= 1u << k;
          else { cfl &= ~(3ull << (2*(sh+k))); if( ref ){ c.gst(c.st.cf, 3*s, 0.0); c.gst(c.st.cf, 3*s+1, 0.0); c.gst(c.st.cf, 3*s+2, 0.0); } }
        }
        while( c.any(in != 0) ){
          if( in == 0 ) continue;
          const int k = RKFD_FFS32(in) - 1; in &= in - 1;
          const int s = pr.sofs + c0 + k, vi = cl.vofs + c0 + k;
          const unsigned long long abit = 1ull << (2*(sh+k)), kbit = 2ull << (2*(sh+k));
          const V3 vw = pw + mul(Rw, v3(m.vert[3*vi], m.vert[3*vi+1], m.vert[3*vi+2]));
          const V3 vb = tmul(Rb, vw - pb);
          V3 n, t1, t2, prob;
          box_face(bx, Rb, vb, bx.half[0]-fabs(vb.x), bx.half[1]-fabs(vb.y), bx.half[2]-fabs(vb.z), n, t1, t2, prob);
          V3 refb;
          if( !(cfl & abit) ){ cfl = (cfl | abit) & ~kbit; refb = prob;
            c.gst(c.st.cref, 3*s, refb.x); c.gst(c.st.cref, 3*s+1, refb.y); c.gst(c.st.cref, 3*s+2, refb.z);
          } else refb = v3(c.gld(c.st.cref,3*s), c.gld(c.st.cref,3*s+1), c.gld(c.st.cref,3*s+2));
          if( pr.type != C_ELASTIC ) continue;     /* rigid pairs are solved by the rigid path */
          const V3 d = vw - (pb + mul(Rb, refb));
          V3 vr = (vlw + cross(omw, vw - pw)) - (vlwB + cross(omwB, vw - pwB));
          if( has_slide(pr) ) vr = vr + slide_vel(m, pr, Rw, pw, RwB, pwB, vw, n);
          V3 f = (-pr.E)*d + (-1.0*(pr.V + pr.E*m.dt))*vr;
          if( dot(f,n) < 0.0 ){ if( ref ){ c.gst(c.st.cf,3*s,f.x); c.gst(c.st.cf,3*s+1,f.y); c.gst(c.st.cf,3*s+2,f.z); } continue; }
          const double fn = dot(f,n), f1 = dot(f,t1), f2 = dot(f,t2);
          const double fs = sqrt(f1*f1 + f2*f2);
          const double mu = (cfl & kbit) ? pr.KF : pr.SF;
          if( !(fabs(fs) < ZTOL) && fs > mu*fn ){
            V3 v = vr + (-dot(vr,n))*n;
            const double vs = norm(v);
            f = fn*n;
            if( !(fabs(vs) < ZTOL) ) f = f + ((-(1.0 - exp(-1.0*m.friction_weight*vs))*pr.KF*fn)/vs)*v;
            if( ref ){ cfl |= kbit; c.gst(c.st.cref,3*s,prob.x); c.gst(c.st.cref,3*s+1,prob.y); c.gst(c.st.cref,3*s+2,prob.z); }
          } else if( ref ){
            cfl &= ~kbit;
            if( has_slide(pr) ){ const V3 nr = refb + slide_ref_shift(m, pr, Rw, pw, RwB, pwB, Rb, vw, n);
              c.gst(c.st.cref,3*s,nr.x); c.gst(c.st.cref,3*s+1,nr.y); c.gst(c.st.cref,3*s+2,nr.z); }
          }
          { const V3 pos = tmul(Rw, vw - pw), fl = tmul(Rw, f); wA.l = wA.l + fl; wA.a = wA.a + cross(pos, fl); }
          { const V3 pos = tmul(RwB, vw - pwB), fl = tmul(RwB, v3(-f.x, -f.y, -f.z)); wB.l = wB.l + fl; wB.a = wB.a + cross(pos, fl); }
          if( ref ){ c.gst(c.st.cf,3*s,f.x); c.gst(c.st.cf,3*s+1,f.y); c.gst(c.st.cf,3*s+2,f.z); }
        }
      }
      c.S(wa) += wA.l.x; c.S(wa+1) += wA.l.y; c.S(wa+2) += wA.l.z; c.S(wa+3) += wA.a.x; c.S(wa+4) += wA.a.y; c.S(wa+5) += wA.a.z;
      c.S(wb) += wB.l.x; c.S(wb+1) += wB.l.y; c.S(wb+2) += wB.l.z; c.S(wb+3) += wB.a.x; c.S(wb+4) += wB.a.y; c.S(wb+5) += wB.a.z;
    }
  }

  /* ---- pass 1: outward kinematics + collision + penalty */
  /* Worlds without rigid pairs: gravity enters as the acceleration (0,0,+g) of the root's parent instead of a force at
   * every centre of mass (same q''; the true link accelerations, which only the rigid-contact solve needs, are
   * not formed): no gravity direction to propagate outward, no gravity terms in the bias forces. */
  static RKFD_HD bool grav_acc(const ModelDev &m){ return Spec::NL != 0 ? true : !m.has_rigid; }

  /* pass-1 values carried outward: world frame, linear velocity (link axes) and angular velocity of the parent link, gravity direction */
  struct Kin { M3 Rw; V3 pw, vl, om, gd; };
  static RKFD_HD void kin_init(Kin &k){ k.Rw = ident3(); k.pw = v3(0,0,0); k.vl = v3(0,0,0); k.om = v3(0,0,0); k.gd = v3(0,0,-GRAVITY); }
  /* sin, cos and velocity of revolute joint i from the T space.  `fresh`: sin/cos are computed from the stage angle (first
   * stage of a step, single evaluations) and stored for the passes that follow; otherwise pass 3 of the previous stage has
   * already rotated them to the new stage angle */
  RKFD_HD void revol_state(const ModelDev &m, int i, bool fresh, double &sn, double &co, double &wz){
    const LinkDev &L = m.link[i]; const int qo = Spec::qofs(i,L);
    if( fresh ){ sincos(T(rk0+qo), &sn, &co); Qw(Spec::sc(i,L), sn); Qw(Spec::sc(i,L)+1, co); }
    else Q2(Spec::sc(i,L), sn, co);
    wz = T(rk0 + Spec::nq(m) + qo);
  }
  /* pass 1 at link i.  A revolute joint's (sin, cos, q') are handed in by the caller (revol_state, or pass 3 of the previous
   * stage in Core::outward).  `cont`: the contacts of the link's cells run here (false: the caller runs them after the loop) */
  template <class Kt>
  RKFD_HD void pass1_link(const ModelDev &m, int i, Kin &k, bool ref, double sn, double co, double wz, bool cont){
    const bool gacc = grav_acc(m);
    const int qs = rk0, qds = rk0 + Spec::nq(m);
    const LinkDev &L = m.link[i]; const int sl = Spec::slot(i,L), qo = Spec::qofs(i,L);
    if( !SER<Kt>(i,L) ){
      if( ROOT<Kt>(i,L) ) kin_init(k);
      else {
        const LinkDev &P = m.link[L.parent];
        k.om = ld3(P.wslot); k.gd = ld3(P.wslot+3);
        if( m.need_world ){ k.Rw = ldm(P.branch_slot); k.pw = ld3(P.branch_slot+9); k.vl = ld3(P.branch_slot+12); }
      }
    }
    XF x; x.fast = 0; x.cls = CLS<Kt>(i,L); x.sg = ro_sign(x.cls, L.rsg); x.c = 1.0; x.s = 0.0;
    x.pz = L.pz;      /* revolute / fixed joint with org position (0, 0, z): decided once on the host (rkfd_model.cpp) */
    V3 vJ = v3(0,0,0), wJ = v3(0,0,0);
    switch(JT<Kt>(i,L)){
    case J_REVOL: {
      x.s = sn; x.c = co; x.p = org_p(L);
      if( CLS<Kt>(i,L) != RO_GENERAL ) x.fast = 1;
      else { const M3 Ro = org_R(L); const V3 o0 = col0(Ro), o1 = col1(Ro);
        x.R = from_cols(co*o0 + sn*o1, co*o1 - sn*o0, col2(Ro)); }
      wJ.z = wz;
    } break;
    case J_PRISM: x.R = org_R(L); x.p = org_p(L) + T(qs+qo)*col2(x.R); vJ.z = T(qds+qo); break;
    case J_SPHER: {
      const M3 Ro = org_R(L);
      x.R = mm(Ro, aa_to_mat(t3(qs+qo))); x.p = org_p(L);
      stm(sl+27, x.R);
      wJ = tmul(x.R, mul(Ro, t3(qds+qo)));
    } break;
    case J_FLOAT: {
      const M3 Ro = org_R(L);
      x.R = mm(Ro, aa_to_mat(t3(qs+qo+3))); x.p = org_p(L) + mul(Ro, t3(qs+qo));
      stm(sl+6, x.R); st3(sl+15, x.p);
      vJ = tmul(x.R, mul(Ro, t3(qds+qo))); wJ = tmul(x.R, mul(Ro, t3(qds+qo+3)));
    } break;
    case J_BRFLOAT: {
      const M3 Ro = org_R(L); const bool brk = (piv >> qo) & 1u;
      x.R = mm(Ro, aa_to_mat(t3(qs+qo+3))); x.p = org_p(L) + mul(Ro, t3(qs+qo));
      stm(sl+6, x.R); st3(sl+15, x.p); c.S(sl+45) = brk ? 1.0 : 0.0;
      const V3 v = t3(qds+qo), w = t3(qds+qo+3);
      if( brk ){ vJ = tmul(x.R, mul(Ro, v)); wJ = tmul(x.R, mul(Ro, w)); }
    } break;
    case J_CYLIN: {
      const M3 Ro = org_R(L); double s1, c1; sincos(T(qs+qo+1), &s1, &c1);
      const V3 o0 = col0(Ro), o1 = col1(Ro);
      x.R = from_cols(c1*o0 + s1*o1, c1*o1 - s1*o0, col2(Ro)); x.p = org_p(L) + T(qs+qo)*col2(Ro);
      stm(sl+17, x.R); st3(sl+26, x.p);
      vJ.z = T(qds+qo); wJ.z = T(qds+qo+1);
    } break;
    case J_HOOKE: {
      const M3 Ro = org_R(L); double s0, c0, s1, c1; sincos(T(qs+qo), &s0, &c0); sincos(T(qs+qo+1), &s1, &c1);
      M3 RJ; RJ.xx = c0*c1; RJ.xy = -s0; RJ.xz = c0*s1; RJ.yx = s0*c1; RJ.yy = c0; RJ.yz = s0*s1; RJ.zx = -s1; RJ.zy = 0.0; RJ.zz = c1;
      x.R = mm(Ro, RJ); x.p = org_p(L);
      stm(sl+17, x.R); st3(sl+26, x.p); c.S(sl+29) = s1; c.S(sl+30) = c1;
      const double v0 = T(qds+qo), v1 = T(qds+qo+1); wJ = v3(-s1*v0, v1, c1*v0);
    } break;
    default: x.R = org_R(L); x.p = org_p(L); break;
    }
    V3 om_n = xf_tmul(x, k.om);
    if( JT<Kt>(i,L) == J_REVOL ) om_n.z += wJ.z; else om_n = om_n + wJ;      /* additions of literal zeros are not folded away */
    if( m.need_world ){
      V3 vl_n = xf_tmul(x, cadd_p(k.vl, k.om, x.p, x.pz));
      if( JT<Kt>(i,L) != J_REVOL ) vl_n = vl_n + vJ;
      k.pw = madd_p(k.pw, k.Rw, x.p, x.pz); k.Rw = xf_world(x, k.Rw); k.vl = vl_n;
    }
    k.om = om_n;
    st3(Spec::wslot(i,L), k.om);
    if( !gacc ){ k.gd = xf_tmul(x, k.gd); st3(Spec::wslot(i,L)+3, k.gd); }
    const int wx = Spec::wext_slot(i,L), fs = Spec::frame_slot(i,L), bs = Spec::branch_slot(i,L), fr = Spec::fext_row(i,L);
    if( cont && wx >= 0 ){
      /* contacts() holds warp votes: a link that only takes an external wrench does not enter it (fr is a compile-time -1 in the
       * specialisations, where this stays the unconditional call) */
      V6 w; w.l = v3(0,0,0); w.a = v3(0,0,0);
      if( fr < 0 || L.cell_end > L.cell_begin ) w = contacts(m, L, k.Rw, k.pw, k.vl, k.om, ref);
      if( fr >= 0 ){
        /* external wrench (force at the centre of mass, torque about it, world axes) -> link axes, about the link origin */
        const V3 f = v3(c.gld(c.st.fext, 6*fr), c.gld(c.st.fext, 6*fr+1), c.gld(c.st.fext, 6*fr+2));
        const V3 n = v3(c.gld(c.st.fext, 6*fr+3), c.gld(c.st.fext, 6*fr+4), c.gld(c.st.fext, 6*fr+5));
        const V3 fl = tmul(k.Rw, f);
        w.l = w.l + fl; w.a = w.a + ( tmul(k.Rw, n) + cross(v3(L.com[0], L.com[1], L.com[2]), fl) );
      }
      st3(wx, w.l); st3(wx+3, w.a);
      if( fs >= 0 ){ stm(fs, k.Rw); st3(fs+9, k.pw); st3(fs+12, k.vl); st3(fs+15, k.om); }
    }
    if( bs >= 0 && m.need_world ){ stm(bs, k.Rw); st3(bs+9, k.pw); st3(bs+12, k.vl); }
  }
  /* `fresh`: as in revol_state */
  RKFD_HD void pass1(const ModelDev &m, bool ref, bool fresh){
    Kin k; kin_init(k);
    auto body = [&](const int i, auto Ktag){
      using Kt = decltype(Ktag);
      if( !Ctx::RIGID ) c.phase_sync(3);
      double sn = 0.0, co = 1.0, wz = 0.0;
      if( JT<Kt>(i, m.link[i]) == J_REVOL ) revol_state(m, i, fresh, sn, co, wz);
      pass1_link<Kt>(m, i, k, ref, sn, co, wz, true);
    };
    links_fwd(m, body);
  }

  /* motor + joint friction of a 1-DoF joint: returns tau = driving torque + friction, jm = rotor inertia
   * (rkfd_util.c:330-364, [EXT A-6, A-7]); at the reference stage commits pivot type and prev_trq */
  /* v = the joint velocity (the caller has it from joint_xform) */
  RKFD_HD double joint_torque(const ModelDev &m, const LinkDev &L, int i, bool ref, double &jm, double u_in, double prev_in, double v){
    const int j = Spec::qofs(i,L);
    const double qj = L.stiffness != 0.0 ? T(rk0 + j) : 0.0;      /* warp-uniform condition: T-space reads stay collective */
    double tdrive = 0.0, tf = 0.0; jm = 0.0;
    if( L.mtype != M_NONE ){
      double e = u_in;
      e = e < L.m_min ? L.m_min : ( e > L.m_max ? L.m_max : e );
      if( L.mtype == M_DC ){
        const double tin = L.m_tin*e, treg = L.m_reg*v;
        jm = L.m_jm; tdrive = tin - treg;
        tf = jm; tf *= -v * m.inv_dt; tf -= tin; tf += treg; tf += prev_in;
        /* static / kinetic bound and the clamp as selects: the lanes of a warp differ in both, and the branches cost more than
         * the three multiply-adds of the kinetic bound (same values as the branching form, bit for bit) */
        const bool kin = (piv >> j) & 1u;
        const double sg = v > 0 ? 1.0 : ( v < 0 ? -1.0 : 0.0 );
        const double fk = fabs(-L.stiffness*qj - L.viscosity*v - L.coulomb*sg);
        const double fmax = kin ? fk : fabs(L.sfriction);
        const bool over = fabs(tf) > fmax;
        tf = over ? ( tf > 0 ? fmax : -fmax ) : tf;
        if( ref ) piv = over ? ( piv | (1u<<j) ) : ( piv & ~(1u<<j) );
      } else tdrive = e;
    }
    if( ref ) c.gst(c.st.piv_prev, j, tdrive + tf);     /* rkFDUpdateJointPrevDrivingTrq (rkfd_util.c:289-311) */
    return tdrive + tf;
  }

  /* ---- pass 2: inward articulated-inertia pass */
  RKFD_HD void pass2(const ModelDev &m, bool ref){
    S3 kA, kC; M3 kB; V3 kf, kn;          /* contribution carried to link i from its serial child */
    kA.xx=kA.xy=kA.xz=kA.yy=kA.yz=kA.zz=0; kC = kA; kB.xx=kB.xy=kB.xz=kB.yx=kB.yy=kB.yz=kB.zx=kB.zy=kB.zz=0; kf = v3(0,0,0); kn = kf;
    const int NLc = Spec::nl(m);
#pragma unroll (Spec::UNROLL)
    for(int i=0;i<NLc;i++) if( Spec::accum_slot(i,m.link[i]) >= 0 ) for(int k=0;k<ACCUM_SLOTS;k++) c.S(m.link[i].accum_slot+k) = 0.0;
    /* motor input and previous driving torque of the NEXT link to be processed are requested one iteration
     * ahead, so that their HBM/L2 latency overlaps the articulated-inertia arithmetic of the current link */
    double nx_u = 0.0, nx_prev = 0.0;
    if( NLc > 0 && m.link[NLc-1].mtype != M_NONE ){ nx_u = c.gld(c.st.u, NLc-1); nx_prev = c.gld(c.st.piv_prev, Spec::qofs(NLc-1, m.link[NLc-1])); }
    const bool gacc = grav_acc(m);
    auto body = [&](const int i, auto Ktag){
      using Kt = decltype(Ktag);
      const LinkDev &L = m.link[i]; const int sl = Spec::slot(i,L);
      if( !Ctx::RIGID ) c.phase_sync(3);
      const double pf_u = nx_u, pf_prev = nx_prev;
      if( i > 0 && m.link[i-1].mtype != M_NONE ){ nx_u = c.gld(c.st.u, i-1); nx_prev = c.gld(c.st.piv_prev, Spec::qofs(i-1, m.link[i-1])); }
      const V3 om = ld3(Spec::wslot(i,L));
      const V3 mc = v3(L.mc[0],L.mc[1],L.mc[2]);
      S3 A, C; M3 B;
      A.xx = L.mass; A.xy = 0; A.xz = 0; A.yy = L.mass; A.yz = 0; A.zz = L.mass;
      B.xx = 0; B.xy = mc.z; B.xz = -mc.y; B.yx = -mc.z; B.yy = 0; B.yz = mc.x; B.zx = mc.y; B.zy = -mc.x; B.zz = 0;
      C.xx = L.Io[0]; C.xy = L.Io[1]; C.xz = L.Io[2]; C.yy = L.Io[3]; C.yz = L.Io[4]; C.zz = L.Io[5];
      /* bias ( w x (w x mc) ; w x (Io w) ) minus gravity (m gd ; mc x gd) minus external wrench */
      V3 pf = cross(om, cross(om, mc));
      V3 pn = cross(om, mul(C, om));
      if( !gacc ){ const V3 gd = ld3(Spec::wslot(i,L)+3); pf = pf - L.mass*gd; pn = pn - cross(mc, gd); }
      if( Spec::wext_slot(i,L) >= 0 ){ pf = pf - ld3(Spec::wext_slot(i,L)); pn = pn - ld3(Spec::wext_slot(i,L)+3); }
      if( Spec::accum_slot(i,L) >= 0 ){
        const int a = L.accum_slot; const S3 aA = lds(a), aC = lds(a+15); const M3 aB = ldm(a+6);
        A.xx+=aA.xx; A.xy+=aA.xy; A.xz+=aA.xz; A.yy+=aA.yy; A.yz+=aA.yz; A.zz+=aA.zz;
        C.xx+=aC.xx; C.xy+=aC.xy; C.xz+=aC.xz; C.yy+=aC.yy; C.yz+=aC.yz; C.zz+=aC.zz;
        B.xx+=aB.xx; B.xy+=aB.xy; B.xz+=aB.xz; B.yx+=aB.yx; B.yy+=aB.yy; B.yz+=aB.yz; B.zx+=aB.zx; B.zy+=aB.zy; B.zz+=aB.zz;
        pf = pf + ld3(a+21); pn = pn + ld3(a+24);
      }
      /* rolled loops: every link but the tip has a serial child, and the tip adds the zero carry */
      if( Spec::ROLL != 0 || ( i+1 < NLc && Spec::serial(i+1, m.link[i+1]) ) ){
        A.xx+=kA.xx; A.xy+=kA.xy; A.xz+=kA.xz; A.yy+=kA.yy; A.yz+=kA.yz; A.zz+=kA.zz;
        C.xx+=kC.xx; C.xy+=kC.xy; C.xz+=kC.xz; C.yy+=kC.yy; C.yz+=kC.yz; C.zz+=kC.zz;
        B.xx+=kB.xx; B.xy+=kB.xy; B.xz+=kB.xz; B.yx+=kB.yx; B.yy+=kB.yy; B.yz+=kB.yz; B.zx+=kB.zx; B.zy+=kB.zy; B.zz+=kB.zz;
        pf = pf + kf; pn = pn + kn;
      }
      V3 vJ, wJ;
      const XF x = joint_xform<Kt>(m, L, i, vJ, wJ);
      /* velocity-product acceleration (link frame): parent angular velocity in link axes = om - wJ */
      /* p' = pA + IA zeta */
      if( JT<Kt>(i,L) == J_REVOL ){
        /* revolute: vJ = 0, wJ = (0,0,q'), so zeta_a = (wp.y q', -wp.x q', 0); written out because products with the
         * literal zeros are not folded by the compiler */
        const V3 omp = v3(om.x, om.y, om.z - wJ.z);
        const V3 zl = cross(omp, cross(omp, x.ptl));
        const double zax = omp.y*wJ.z, zay = -omp.x*wJ.z;
        pf = madd(pf, A, zl);
        pf = v3(fma(B.xy,zay,fma(B.xx,zax,pf.x)), fma(B.yy,zay,fma(B.yx,zax,pf.y)), fma(B.zy,zay,fma(B.zx,zax,pf.z)));
        pn = maddt(pn, B, zl);
        pn = v3(fma(C.xy,zay,fma(C.xx,zax,pn.x)), fma(C.yy,zay,fma(C.xy,zax,pn.y)), fma(C.yz,zay,fma(C.xz,zax,pn.z)));
      } else if( JT<Kt>(i,L) != J_FLOAT && !( JT<Kt>(i,L) == J_BRFLOAT && c.S(sl+45) != 0.0 ) ){
        const V3 omp = om - wJ;
        const V3 zl = cross(omp, cross(omp, x.ptl)) + 2.0*cross(omp, vJ);
        V3 za = cross(omp, wJ);
        if( JT<Kt>(i,L) == J_HOOKE ){ const double qq = T(rk0 + Spec::nq(m) + Spec::qofs(i,L))*T(rk0 + Spec::nq(m) + Spec::qofs(i,L) + 1);   /* S' q' */
          za.x -= c.S(sl+30)*qq; za.z -= c.S(sl+29)*qq; }
        pf = madd(madd(pf, A, zl), B, za);
        pn = madd(maddt(pn, B, zl), C, za);
      }
      switch(JT<Kt>(i,L)){
      case J_REVOL: {
        double jm; const double tau = joint_torque(m, L, i, ref, jm, pf_u, pf_prev, wJ.z);
        const V3 Ul = col2(B), Ua = v3(C.xz, C.yz, C.zz);
        const double Dinv = 1.0/(C.zz + jm), u = tau - pn.z;
        st3(sl, Ul); st3(sl+3, Ua); Qw(Spec::sc(i,L)+2, Dinv); Qw(Spec::sc(i,L)+3, u);
        const V3 Wl = Dinv*Ul, Wa = Dinv*Ua;
        A.xx-=Wl.x*Ul.x; A.xy-=Wl.x*Ul.y; A.xz-=Wl.x*Ul.z; A.yy-=Wl.y*Ul.y; A.yz-=Wl.y*Ul.z; A.zz-=Wl.z*Ul.z;
        C.xx-=Wa.x*Ua.x; C.xy-=Wa.x*Ua.y; C.xz-=Wa.x*Ua.z; C.yy-=Wa.y*Ua.y; C.yz-=Wa.y*Ua.z; C.zz-=Wa.z*Ua.z;
        B.xx-=Wl.x*Ua.x; B.xy-=Wl.x*Ua.y; B.xz-=Wl.x*Ua.z; B.yx-=Wl.y*Ua.x; B.yy-=Wl.y*Ua.y; B.yz-=Wl.y*Ua.z; B.zx-=Wl.z*Ua.x; B.zy-=Wl.z*Ua.y; B.zz-=Wl.z*Ua.z;
        pf = vfma(u, Wl, pf); pn = vfma(u, Wa, pn);
      } break;
      case J_PRISM: {
        double jm; const double tau = joint_torque(m, L, i, ref, jm, pf_u, pf_prev, vJ.z);
        const V3 Ul = v3(A.xz, A.yz, A.zz), Ua = v3(B.zx, B.zy, B.zz);
        const double Dinv = 1.0/(A.zz + jm), u = tau - pf.z;
        st3(sl, Ul); st3(sl+3, Ua); Qw(Spec::sc(i,L)+2, Dinv); Qw(Spec::sc(i,L)+3, u);
        const V3 Wl = Dinv*Ul, Wa = Dinv*Ua;
        A.xx-=Wl.x*Ul.x; A.xy-=Wl.x*Ul.y; A.xz-=Wl.x*Ul.z; A.yy-=Wl.y*Ul.y; A.yz-=Wl.y*Ul.z; A.zz-=Wl.z*Ul.z;
        C.xx-=Wa.x*Ua.x; C.xy-=Wa.x*Ua.y; C.xz-=Wa.x*Ua.z; C.yy-=Wa.y*Ua.y; C.yz-=Wa.y*Ua.z; C.zz-=Wa.z*Ua.z;
        B.xx-=Wl.x*Ua.x; B.xy-=Wl.x*Ua.y; B.xz-=Wl.x*Ua.z; B.yx-=Wl.y*Ua.x; B.yy-=Wl.y*Ua.y; B.yz-=Wl.y*Ua.z; B.zx-=Wl.z*Ua.x; B.zy-=Wl.z*Ua.y; B.zz-=Wl.z*Ua.z;
        pf = vfma(u, Wl, pf); pn = vfma(u, Wa, pn);
      } break;
      case J_SPHER: {
        /* S = [0; E], E = R^T Ro (= RJ^T); U = [B E; C E]; D = E^T C E; tau = 0 */
        const M3 E = tmm(x.R, org_R(L));
        const M3 Ul = mm(B, E); M3 Cf; Cf.xx=C.xx; Cf.xy=C.xy; Cf.xz=C.xz; Cf.yx=C.xy; Cf.yy=C.yy; Cf.yz=C.yz; Cf.zx=C.xz; Cf.zy=C.yz; Cf.zz=C.zz;
        const M3 Ua = mm(Cf, E);
        const M3 Df = tmm(E, Ua); S3 D; D.xx=Df.xx; D.xy=Df.xy; D.xz=Df.xz; D.yy=Df.yy; D.yz=Df.yz; D.zz=Df.zz;
        const S3 Di = sym3_inverse(D);
        const V3 u = -tmul(E, pn);
        stm(sl, Ul); stm(sl+9, Ua);
        c.S(sl+18)=Di.xx; c.S(sl+19)=Di.xy; c.S(sl+20)=Di.xz; c.S(sl+21)=Di.yy; c.S(sl+22)=Di.yz; c.S(sl+23)=Di.zz;
        st3(sl+24, u);
        M3 Dif; Dif.xx=Di.xx; Dif.xy=Di.xy; Dif.xz=Di.xz; Dif.yx=Di.xy; Dif.yy=Di.yy; Dif.yz=Di.yz; Dif.zx=Di.xz; Dif.zy=Di.yz; Dif.zz=Di.zz;
        const M3 Wl = mm(Ul, Dif), Wa = mm(Ua, Dif);
        const M3 dA = mm(Wl, transpose(Ul)), dB = mm(Wl, transpose(Ua)), dC = mm(Wa, transpose(Ua));
        A.xx-=dA.xx; A.xy-=dA.xy; A.xz-=dA.xz; A.yy-=dA.yy; A.yz-=dA.yz; A.zz-=dA.zz;
        C.xx-=dC.xx; C.xy-=dC.xy; C.xz-=dC.xz; C.yy-=dC.yy; C.yz-=dC.yz; C.zz-=dC.zz;
        B.xx-=dB.xx; B.xy-=dB.xy; B.xz-=dB.xz; B.yx-=dB.yx; B.yy-=dB.yy; B.yz-=dB.yz; B.zx-=dB.zx; B.zy-=dB.zy; B.zz-=dB.zz;
        pf = pf + mul(Wl, u); pn = pn + mul(Wa, u);
      } break;
      case J_CYLIN: case J_HOOKE: {
        /* two motion axes S_k = (l_k; a_k): U_k = IA S_k, D = S^T U (2x2), u = -S^T pA (no motor, no passive torque:
         * rkFDJointFrictionAll with zero kinetic friction, rkfd_util.c:318-328) */
        V3 l0, a0, l1, a1; axes2(JT<Kt>(i,L), sl, l0, a0, l1, a1);
        const V3 Ul0 = mul(A, l0) + mul(B, a0), Ua0 = tmul(B, l0) + mul(C, a0);
        const V3 Ul1 = mul(A, l1) + mul(B, a1), Ua1 = tmul(B, l1) + mul(C, a1);
        const double d00 = dot(l0,Ul0) + dot(a0,Ua0), d01 = dot(l0,Ul1) + dot(a0,Ua1), d11 = dot(l1,Ul1) + dot(a1,Ua1);
        const double idet = 1.0/(d00*d11 - d01*d01), i00 = d11*idet, i01 = -d01*idet, i11 = d00*idet;
        const double u0 = -(dot(l0,pf) + dot(a0,pn)), u1 = -(dot(l1,pf) + dot(a1,pn));
        st3(sl, Ul0); st3(sl+3, Ua0); st3(sl+6, Ul1); st3(sl+9, Ua1);
        c.S(sl+12) = i00; c.S(sl+13) = i01; c.S(sl+14) = i11; c.S(sl+15) = u0; c.S(sl+16) = u1;
        const V3 Wl0 = i00*Ul0 + i01*Ul1, Wa0 = i00*Ua0 + i01*Ua1, Wl1 = i01*Ul0 + i11*Ul1, Wa1 = i01*Ua0 + i11*Ua1;
        A.xx-=Wl0.x*Ul0.x+Wl1.x*Ul1.x; A.xy-=Wl0.x*Ul0.y+Wl1.x*Ul1.y; A.xz-=Wl0.x*Ul0.z+Wl1.x*Ul1.z; A.yy-=Wl0.y*Ul0.y+Wl1.y*Ul1.y; A.yz-=Wl0.y*Ul0.z+Wl1.y*Ul1.z; A.zz-=Wl0.z*Ul0.z+Wl1.z*Ul1.z;
        C.xx-=Wa0.x*Ua0.x+Wa1.x*Ua1.x; C.xy-=Wa0.x*Ua0.y+Wa1.x*Ua1.y; C.xz-=Wa0.x*Ua0.z+Wa1.x*Ua1.z; C.yy-=Wa0.y*Ua0.y+Wa1.y*Ua1.y; C.yz-=Wa0.y*Ua0.z+Wa1.y*Ua1.z; C.zz-=Wa0.z*Ua0.z+Wa1.z*Ua1.z;
        B.xx-=Wl0.x*Ua0.x+Wl1.x*Ua1.x; B.xy-=Wl0.x*Ua0.y+Wl1.x*Ua1.y; B.xz-=Wl0.x*Ua0.z+Wl1.x*Ua1.z;
        B.yx-=Wl0.y*Ua0.x+Wl1.y*Ua1.x; B.yy-=Wl0.y*Ua0.y+Wl1.y*Ua1.y; B.yz-=Wl0.y*Ua0.z+Wl1.y*Ua1.z;
        B.zx-=Wl0.z*Ua0.x+Wl1.z*Ua1.x; B.zy-=Wl0.z*Ua0.y+Wl1.z*Ua1.y; B.zz-=Wl0.z*Ua0.z+Wl1.z*Ua1.z;
        pf = pf + u0*Wl0 + u1*Wl1; pn = pn + u0*Wa0 + u1*Wa1;
      } break;
      case J_FLOAT:       /* free 6-DoF joint: a = -IA^-1 pA, nothing is transmitted to the parent */
        float_project(A, B, C, pf, pn, sl, m.has_rigid != 0);
        break;
      case J_BRFLOAT:
        if( c.S(sl+45) != 0.0 ) float_project(A, B, C, pf, pn, sl, true);
        else {             /* rigid: everything is handed to the parent; IA and p' are kept for the wrench test of pass 3 */
          c.S(sl+18)=A.xx; c.S(sl+19)=A.xy; c.S(sl+20)=A.xz; c.S(sl+21)=A.yy; c.S(sl+22)=A.yz; c.S(sl+23)=A.zz;
          stm(sl+24, B);
          c.S(sl+33)=C.xx; c.S(sl+34)=C.xy; c.S(sl+35)=C.xz; c.S(sl+36)=C.yy; c.S(sl+37)=C.yz; c.S(sl+38)=C.zz;
          st3(sl+39, pf); st3(sl+42, pn);
        }
        break;
      default: break;
      }
      if( ROOT<Kt>(i,L) || JT<Kt>(i,L) == J_FLOAT ) return;
      if( JT<Kt>(i,L) == J_BRFLOAT && c.S(sl+45) != 0.0 ){    /* a broken joint transmits nothing (the lanes of a warp may differ here) */
        A.xx=A.xy=A.xz=A.yy=A.yz=A.zz=0; C = A; B.xx=B.xy=B.xz=B.yx=B.yy=B.yz=B.zx=B.zy=B.zz=0; pf = v3(0,0,0); pn = pf; }
      /* X^T Ia X and X^T pa into the parent frame */
      const V3 p = x.p;
      const S3 Ar = xf_sym(x, A), Cr = xf_sym(x, C); const M3 Br = xf_gen(x, B);
      const M3 Bp = shift_B_p(Br, Ar, p, x.pz);           /* B_p = B' - A' [p x] */
      const S3 Cp = shift_C_p(Cr, Bp, Br, p, x.pz);       /* C_p = C' + [p x] B_p + ([p x] B')^T */
      const V3 fp = xf_mul(x, pf); const V3 np = padd_c(xf_mul(x, pn), p, fp, x.pz);
      if( SER<Kt>(i,L) ){ kA = Ar; kB = Bp; kC = Cp; kf = fp; kn = np; }
      else {
        const int a = m.link[L.parent].accum_slot;
        c.S(a)+=Ar.xx; c.S(a+1)+=Ar.xy; c.S(a+2)+=Ar.xz; c.S(a+3)+=Ar.yy; c.S(a+4)+=Ar.yz; c.S(a+5)+=Ar.zz;
        c.S(a+6)+=Bp.xx; c.S(a+7)+=Bp.xy; c.S(a+8)+=Bp.xz; c.S(a+9)+=Bp.yx; c.S(a+10)+=Bp.yy; c.S(a+11)+=Bp.yz; c.S(a+12)+=Bp.zx; c.S(a+13)+=Bp.zy; c.S(a+14)+=Bp.zz;
        c.S(a+15)+=Cp.xx; c.S(a+16)+=Cp.xy; c.S(a+17)+=Cp.xz; c.S(a+18)+=Cp.yy; c.S(a+19)+=Cp.yz; c.S(a+20)+=Cp.zz;
        c.S(a+21)+=fp.x; c.S(a+22)+=fp.y; c.S(a+23)+=fp.z; c.S(a+24)+=np.x; c.S(a+25)+=np.y; c.S(a+26)+=np.z;
      }
    };
    links_bwd(m, body);
  }

  /* Runge-Kutta-Gill bookkeeping of one scalar state pair (x, x') with slope (kq, kv) ([EXT A-9]):
   * stage states are built from the committed state by successive increments, the combination is
   * accumulated in the output buffer */
  /* The other explicit schemes of [EXT] zODE2AssignRegular use the same bookkeeping: classical Runge-Kutta is the
   * same four stages with c31 = c42 = 0; Heun runs stages K1 and K4 (c21 = dt, b1 = b4 = dt/2); Euler runs K1 alone,
   * whose running combination is already the new state (ns = 1). */
  using RK = ModelDev::RK;
  static RKFD_HD int rk_stages(int integrator){ return integrator == 2 ? 1 : ( integrator == 3 ? 2 : 4 ); }
  static RKFD_HD int rk_next_stage(int stage, int ns){ return stage == ST_K1 ? ( ns == 4 ? ST_K2 : ( ns == 2 ? ST_K4 : ST_REF ) ) : stage + 1; }
  /* velocity-like (vector-space) component j */
  RKFD_HD void rk_lin(const ModelDev &m, const RK &k, int stage, int slotS, int slotP, double *gin, double *gout, int j, double slope){
    const double F = ( stage >= ST_K2 && stage <= ST_K4 ) ? c.gld(gout, j) : 0.0, x0 = stage == ST_K2 ? c.gld(gin, j) : 0.0;
    rk_lin_pf(k, stage, slotS, slotP, gout, j, slope, F, x0, stage == ST_K1 ? T(slotS) : 0.0);
  }
  /* F = running combination and x0 = committed value, fetched by the caller (possibly one link ahead); xs = the stage value
   * (T space slotS) at stage K1, which the caller has already loaded */
  RKFD_HD double rk_lin_pf(const RK &k, int stage, int slotS, int slotP, double *gout, int j, double slope, double F, double x0g, double xs){
    double xn = 0.0;       /* the next stage value */
    switch(stage){
    case ST_K1: { const double x0 = xs; const double F = x0 + k.b1*slope; c.gst(gout, j, F); Tw(slotP, x0 + k.c31*slope); xn = k.ns == 1 ? F : x0 + k.c21*slope; Tw(slotS, xn); } break;
    case ST_K2: { c.gst(gout, j, F + k.b2*slope); xn = T(slotP) + k.c32*slope; Tw(slotS, xn); Tw(slotP, x0g + k.c42*slope); } break;
    case ST_K3: { c.gst(gout, j, F + k.b3*slope); xn = T(slotP) + k.c43*slope; Tw(slotS, xn); } break;
    case ST_K4: { xn = F + k.b4*slope; c.gst(gout, j, xn); Tw(slotS, xn); } break;
    default: break;
    }
    return xn;
  }
  /* sin/cos of a revolute joint carried from the stage angle qold to qnew = qold + d: angle addition with the
   * Taylor series of (sin d, cos d) (|d| <= 1/16: truncation below 1e-18), a full sincos otherwise.  A step
   * computes sincos once per joint (first stage) instead of five times; four chained rotations add a few ulp. */
  RKFD_HD void rot_sincos(const ModelDev &m, int sc, double s0, double c0, double qold, double qnew, double &sn, double &co){
    const double d = qnew - qold, d2 = d*d;
    /* the coefficients 1/9!, -1/7!, 1/5!, -1/3!, 1/8!, -1/6! come from the model table (same values: operands of the multiply-adds
     * instead of two moves each) */
    const double sd = d*fma(d2, fma(d2, fma(d2, fma(d2, m.tay[0], m.tay[1]), m.tay[2]), m.tay[3]), 1.0);
    const double cd = fma(d2, fma(d2, fma(d2, fma(d2, m.tay[4], m.tay[5]), 1.0/24.0), -0.5), 1.0);
    sn = fma(s0, cd, c0*sd); co = fma(c0, cd, -(s0*sd));
    if( !(fabs(d) <= 0.0625) ) sincos(qnew, &sn, &co);
    Qw(sc, sn); Qw(sc+1, co);
  }
  /* rotation (angle-axis) component triple starting at j: increments compose on SO(3) */
  RKFD_HD void rk_rot(const ModelDev &m, const RK &k, int stage, int slotS, int slotP, double *gin, double *gout, int j, V3 w){
    switch(stage){
    case ST_K1: { const V3 x0 = t3(slotS); const V3 F = aa_cascade(x0, k.b1*w);
      c.gst(gout,j,F.x); c.gst(gout,j+1,F.y); c.gst(gout,j+2,F.z);
      tw3(slotP, k.c31 == 0.0 ? x0 : aa_cascade(x0, k.c31*w)); tw3(slotS, k.ns == 1 ? F : aa_cascade(x0, k.c21*w)); } break;
    case ST_K2: { const V3 x0 = v3(c.gld(gin,j), c.gld(gin,j+1), c.gld(gin,j+2));
      const V3 F = aa_cascade(v3(c.gld(gout,j), c.gld(gout,j+1), c.gld(gout,j+2)), k.b2*w);
      c.gst(gout,j,F.x); c.gst(gout,j+1,F.y); c.gst(gout,j+2,F.z);
      tw3(slotS, aa_cascade(t3(slotP), k.c32*w)); tw3(slotP, k.c42 == 0.0 ? x0 : aa_cascade(x0, k.c42*w)); } break;
    case ST_K3: { const V3 F = aa_cascade(v3(c.gld(gout,j), c.gld(gout,j+1), c.gld(gout,j+2)), k.b3*w);
      c.gst(gout,j,F.x); c.gst(gout,j+1,F.y); c.gst(gout,j+2,F.z);
      tw3(slotS, aa_cascade(t3(slotP), k.c43*w)); } break;
    case ST_K4: { const V3 F = aa_cascade(v3(c.gld(gout,j), c.gld(gout,j+1), c.gld(gout,j+2)), k.b4*w);
      c.gst(gout,j,F.x); c.gst(gout,j+1,F.y); c.gst(gout,j+2,F.z); tw3(slotS, F); } break;
    default: break;
    }
  }
  /* one dof: displacement uses the stage velocity as slope, velocity uses the acceleration */
  RKFD_HD void rk_dof(const ModelDev &m, const RK &k, int stage, int j, double acc){
    const int qs = rk0 + j, qds = rk0 + m.nq + j, pq = rk0 + 2*m.nq + j, pqd = rk0 + 3*m.nq + j;
    if( stage == ST_PROBE ) return;
    if( stage >= ST_REF ){ c.gst(c.st.qdd, j, acc); if( !(fabs(acc) < 1.0e300) ) bad = 1; return; }
    const double vel = T(qds);
    rk_lin(m, k, stage, qs, pq, qc, qn, j, vel);
    rk_lin(m, k, stage, qds, pqd, qdc, qdn, j, acc);
  }

  /* ---- pass 3: outward acceleration pass + integrator bookkeeping */
  /* pass-3 values carried outward: linear / angular acceleration and angular velocity of the parent link; the running
   * combination (and, at stage 2, the committed state) of the next 1-DoF joint, requested one link ahead */
  struct Acc { V3 al, aa, om; double nxq[4]; };
  static RKFD_HD void acc_init(Acc &a){ a.al = v3(0,0,0); a.aa = v3(0,0,0); a.om = v3(0,0,0); a.nxq[0] = a.nxq[1] = a.nxq[2] = a.nxq[3] = 0; }
  /* pass 3 at link i.  Stages K1-K4: a revolute joint returns its (sin, cos, q') of the next stage in (sn, co, wz), the
   * values it also stores in the T space */
  template <class Kt>
  RKFD_HD void pass3_link(const ModelDev &m, int i, Acc &a, int stage, double &sn, double &co, double &wz){
    const RK &k = m.rk;
    const bool pfF = stage >= ST_K2 && stage <= ST_K4, pfX = stage == ST_K2;
    const int NLc = Spec::nl(m), NQc = Spec::nq(m);
    const LinkDev &L = m.link[i]; const int sl = Spec::slot(i,L), qo = Spec::qofs(i,L);
    if( i == 0 && Spec::ndof(i,L) == 1 ){
      if( pfF ){ a.nxq[0] = c.gld(qn, qo); a.nxq[1] = c.gld(qdn, qo); }
      if( pfX ){ a.nxq[2] = c.gld(qc, qo); a.nxq[3] = c.gld(qdc, qo); }
    }
    const double pfq[4] = { a.nxq[0], a.nxq[1], a.nxq[2], a.nxq[3] };
    if( i+1 < NLc && Spec::ndof(i+1, m.link[i+1]) == 1 ){
      const int jn = Spec::qofs(i+1, m.link[i+1]);
      if( pfF ){ a.nxq[0] = c.gld(qn, jn); a.nxq[1] = c.gld(qdn, jn); }
      if( pfX ){ a.nxq[2] = c.gld(qc, jn); a.nxq[3] = c.gld(qdc, jn); }
    }
    if( !SER<Kt>(i,L) ){
      if( ROOT<Kt>(i,L) ){ a.al = v3(0,0, grav_acc(m) ? GRAVITY : 0.0); a.aa = v3(0,0,0); a.om = v3(0,0,0); }
      else { const int b = m.link[L.parent].branch_slot; a.al = ld3(b); a.aa = ld3(b+3); a.om = ld3(b+6); }
    }
    V3 vJ, wJ;
    const XF x = joint_xform<Kt>(m, L, i, vJ, wJ);
    const V3 omp = xf_tmul(x, a.om);
    V3 zl, za;
    if( JT<Kt>(i,L) == J_REVOL ){ zl = cross(omp, cross(omp, x.ptl)); za = v3(omp.y*wJ.z, -omp.x*wJ.z, 0.0); }
    else { zl = cross(omp, cross(omp, x.ptl)) + 2.0*cross(omp, vJ); za = cross(omp, wJ); }
    const V3 xl = xf_tmul(x, cadd_p(a.al, a.aa, x.p, x.pz)), xa = xf_tmul(x, a.aa);
    switch(JT<Kt>(i,L)){
    case J_REVOL: case J_PRISM: {
      const V3 Ul = ld3(sl), Ua = ld3(sl+3);
      double Dinv, uu; Q2(Spec::sc(i,L)+2, Dinv, uu);
      const double acc = Dinv*fma(-Ua.z,xa.z,fma(-Ua.y,xa.y,fma(-Ua.x,xa.x,fma(-Ul.z,xl.z,fma(-Ul.y,xl.y,fma(-Ul.x,xl.x,uu))))));
      if( JT<Kt>(i,L) == J_REVOL ){
        a.al = cadd(xl, omp, cross(omp, x.ptl));
        a.aa = v3(fma(omp.y, wJ.z, xa.x), fma(-omp.x, wJ.z, xa.y), xa.z + acc);
      } else { a.al = xl + zl; a.aa = xa + za; a.al.z += acc; }
      if( stage == ST_PROBE ){}
      else if( stage >= ST_REF ){ c.gst(c.st.qdd, qo, acc); if( !(fabs(acc) < 1.0e300) ) bad = 1; }
      else {
        const int j = qo, qs = rk0 + j, qds = qs + NQc, pq = qs + 2*NQc, pqd = qs + 3*NQc;
        const double vel = JT<Kt>(i,L) == J_REVOL ? wJ.z : vJ.z;     /* T(qds), loaded by joint_xform */
        const double qold = ( JT<Kt>(i,L) == J_REVOL || stage == ST_K1 ) ? T(qs) : 0.0;
        const double qnew = rk_lin_pf(k, stage, qs,  pq,  qn,  j, vel, pfq[0], pfq[2], qold);
        if( JT<Kt>(i,L) == J_REVOL ) rot_sincos(m, Spec::sc(i,L), x.s, x.c, qold, qnew, sn, co);
        wz = rk_lin_pf(k, stage, qds, pqd, qdn, j, acc, pfq[1], pfq[3], vel);
      }
    } break;
    case J_SPHER: {
      const M3 Ul = ldm(sl), Ua = ldm(sl+9); const S3 Di = lds(sl+18); const V3 u = ld3(sl+24);
      const V3 rhs = u - (tmul(Ul, xl) + tmul(Ua, xa));
      const V3 acc = mul(Di, rhs);
      const M3 E = tmm(x.R, org_R(L));
      a.al = xl + zl; a.aa = xa + za + mul(E, acc);
      if( stage == ST_PROBE ){}
      else if( stage >= ST_REF ){ c.gst(c.st.qdd,L.qofs,acc.x); c.gst(c.st.qdd,L.qofs+1,acc.y); c.gst(c.st.qdd,L.qofs+2,acc.z);
        if( !(fabs(acc.x)+fabs(acc.y)+fabs(acc.z) < 1.0e300) ) bad = 1; }
      else {
        const int qs = rk0 + L.qofs, qds = qs + m.nq, pq = qs + 2*m.nq, pqd = qs + 3*m.nq;
        const V3 w = t3(qds);
        rk_rot(m, k, stage, qs, pq, qc, qn, L.qofs, w);
        rk_lin(m, k, stage, qds,   pqd,   qdc, qdn, L.qofs,   acc.x);
        rk_lin(m, k, stage, qds+1, pqd+1, qdc, qdn, L.qofs+1, acc.y);
        rk_lin(m, k, stage, qds+2, pqd+2, qdc, qdn, L.qofs+2, acc.z);
      }
    } break;
    case J_CYLIN: case J_HOOKE: {
      if( JT<Kt>(i,L) == J_HOOKE ){ const double qq = T(rk0 + NQc + qo)*T(rk0 + NQc + qo + 1); za.x -= c.S(sl+30)*qq; za.z -= c.S(sl+29)*qq; }
      V3 l0, a0, l1, a1; axes2(JT<Kt>(i,L), sl, l0, a0, l1, a1);
      const double r0 = c.S(sl+15) - (dot(ld3(sl),xl) + dot(ld3(sl+3),xa)), r1 = c.S(sl+16) - (dot(ld3(sl+6),xl) + dot(ld3(sl+9),xa));
      const double acc0 = c.S(sl+12)*r0 + c.S(sl+13)*r1, acc1 = c.S(sl+13)*r0 + c.S(sl+14)*r1;
      a.al = xl + zl + acc0*l0 + acc1*l1; a.aa = xa + za + acc0*a0 + acc1*a1;
      if( stage == ST_PROBE ){}
      else if( stage >= ST_REF ){ c.gst(c.st.qdd, qo, acc0); c.gst(c.st.qdd, qo+1, acc1); if( !(fabs(acc0)+fabs(acc1) < 1.0e300) ) bad = 1; }
      else {
        const int qs = rk0 + qo, qds = qs + m.nq, pq = qs + 2*m.nq, pqd = qs + 3*m.nq;
        const double v0 = T(qds), v1 = T(qds+1);
        rk_lin(m, k, stage, qs,   pq,   qc, qn, qo,   v0);
        rk_lin(m, k, stage, qs+1, pq+1, qc, qn, qo+1, v1);
        rk_lin(m, k, stage, qds,   pqd,   qdc, qdn, qo,   acc0);
        rk_lin(m, k, stage, qds+1, pqd+1, qdc, qdn, qo+1, acc1);
      }
    } break;
    case J_FLOAT: {
      const V3 a0l = ld3(sl), a0a = ld3(sl+3);
      const M3 RJ = mm(transpose(org_R(L)), x.R);     /* S^-1 = blockdiag(RJ, RJ) */
      const V3 accl = mul(RJ, a0l - xl - zl), acca = mul(RJ, a0a - xa - za);
      a.al = a0l; a.aa = a0a;
      if( stage == ST_PROBE ){}
      else if( stage >= ST_REF ){
        c.gst(c.st.qdd,L.qofs,accl.x); c.gst(c.st.qdd,L.qofs+1,accl.y); c.gst(c.st.qdd,L.qofs+2,accl.z);
        c.gst(c.st.qdd,L.qofs+3,acca.x); c.gst(c.st.qdd,L.qofs+4,acca.y); c.gst(c.st.qdd,L.qofs+5,acca.z);
        if( !(fabs(accl.x)+fabs(accl.y)+fabs(accl.z)+fabs(acca.x)+fabs(acca.y)+fabs(acca.z) < 1.0e300) ) bad = 1;
      } else {
        const int qs = rk0 + L.qofs, qds = qs + m.nq, pq = qs + 2*m.nq, pqd = qs + 3*m.nq;
        const V3 v = t3(qds), w = t3(qds+3);
        rk_lin(m, k, stage, qs,   pq,   qc, qn, L.qofs,   v.x);
        rk_lin(m, k, stage, qs+1, pq+1, qc, qn, L.qofs+1, v.y);
        rk_lin(m, k, stage, qs+2, pq+2, qc, qn, L.qofs+2, v.z);
        rk_rot(m, k, stage, qs+3, pq+3, qc, qn, L.qofs+3, w);
        rk_lin(m, k, stage, qds,   pqd,   qdc, qdn, L.qofs,   accl.x);
        rk_lin(m, k, stage, qds+1, pqd+1, qdc, qdn, L.qofs+1, accl.y);
        rk_lin(m, k, stage, qds+2, pqd+2, qdc, qdn, L.qofs+2, accl.z);
        rk_lin(m, k, stage, qds+3, pqd+3, qdc, qdn, L.qofs+3, acca.x);
        rk_lin(m, k, stage, qds+4, pqd+4, qdc, qdn, L.qofs+4, acca.y);
        rk_lin(m, k, stage, qds+5, pqd+5, qdc, qdn, L.qofs+5, acca.z);
      }
    } break;
    case J_BRFLOAT: {
      /* broken: the float joint; rigid: the fixed joint whose six dofs are held (zero slopes), and in the committing
       * evaluation the wrench it transmits, IA (X a_parent) + p' at the link origin ([EXT A-17]; rkChainUpdateABIWrench,
       * rkfd_sim.c:511-514), is compared with its thresholds.  One code path for both: the integrator bookkeeping touches
       * the T space, which only warp-uniform code may do. */
      const bool brk = c.S(sl+45) != 0.0;
      V3 accl = v3(0,0,0), acca = v3(0,0,0);
      if( brk ){ const V3 a0l = ld3(sl), a0a = ld3(sl+3); const M3 RJ = mm(transpose(org_R(L)), x.R);
        accl = mul(RJ, a0l - xl - zl); acca = mul(RJ, a0a - xa - za); a.al = a0l; a.aa = a0a; }
      else { a.al = xl + zl; a.aa = xa + za; }
      if( stage == ST_PROBE ){}
      else if( stage >= ST_REF ){
        c.gst(c.st.qdd,L.qofs,accl.x); c.gst(c.st.qdd,L.qofs+1,accl.y); c.gst(c.st.qdd,L.qofs+2,accl.z);
        c.gst(c.st.qdd,L.qofs+3,acca.x); c.gst(c.st.qdd,L.qofs+4,acca.y); c.gst(c.st.qdd,L.qofs+5,acca.z);
        if( !(fabs(accl.x)+fabs(accl.y)+fabs(accl.z)+fabs(acca.x)+fabs(acca.y)+fabs(acca.z) < 1.0e300) ) bad = 1;
        if( !brk && ( stage == ST_REF || stage == ST_EVAL_REF ) ){
          S3 A, C; A.xx=c.S(sl+18); A.xy=c.S(sl+19); A.xz=c.S(sl+20); A.yy=c.S(sl+21); A.yz=c.S(sl+22); A.zz=c.S(sl+23);
          const M3 B = ldm(sl+24);
          C.xx=c.S(sl+33); C.xy=c.S(sl+34); C.xz=c.S(sl+35); C.yy=c.S(sl+36); C.yz=c.S(sl+37); C.zz=c.S(sl+38);
          const V3 f = ld3(sl+39) + mul(A, xl) + mul(B, xa), n = ld3(sl+42) + tmul(B, xl) + mul(C, xa);
          if( norm(f) > L.brk_f || norm(n) > L.brk_t ) piv |= 1u << L.qofs;
        }
      } else {
        const int qs = rk0 + L.qofs, qds = qs + m.nq, pq = qs + 2*m.nq, pqd = qs + 3*m.nq;
        V3 v = t3(qds), w = t3(qds+3);
        if( !brk ){ v = v3(0,0,0); w = v; }
        rk_lin(m, k, stage, qs,   pq,   qc, qn, L.qofs,   v.x);
        rk_lin(m, k, stage, qs+1, pq+1, qc, qn, L.qofs+1, v.y);
        rk_lin(m, k, stage, qs+2, pq+2, qc, qn, L.qofs+2, v.z);
        rk_rot(m, k, stage, qs+3, pq+3, qc, qn, L.qofs+3, w);
        rk_lin(m, k, stage, qds,   pqd,   qdc, qdn, L.qofs,   accl.x);
        rk_lin(m, k, stage, qds+1, pqd+1, qdc, qdn, L.qofs+1, accl.y);
        rk_lin(m, k, stage, qds+2, pqd+2, qdc, qdn, L.qofs+2, accl.z);
        rk_lin(m, k, stage, qds+3, pqd+3, qdc, qdn, L.qofs+3, acca.x);
        rk_lin(m, k, stage, qds+4, pqd+4, qdc, qdn, L.qofs+4, acca.y);
        rk_lin(m, k, stage, qds+5, pqd+5, qdc, qdn, L.qofs+5, acca.z);
      }
    } break;
    default: a.al = xl + zl; a.aa = xa + za; break;
    }
    if( JT<Kt>(i,L) == J_REVOL ) a.om = v3(omp.x, omp.y, omp.z + wJ.z); else a.om = omp + wJ;
    if( Spec::frame_slot(i,L) >= 0 ){ st3(Spec::frame_slot(i,L)+18, a.al); st3(Spec::frame_slot(i,L)+21, a.aa); }
    if( Spec::branch_slot(i,L) >= 0 ){ st3(L.branch_slot, a.al); st3(L.branch_slot+3, a.aa); st3(L.branch_slot+6, a.om); }
  }
  RKFD_HD void pass3(const ModelDev &m, int stage){
    Acc a; acc_init(a);
    auto body = [&](const int i, auto Ktag){
      using Kt = decltype(Ktag);
      if( !Ctx::RIGID ) c.phase_sync(3);
      double sn, co, wz;
      pass3_link<Kt>(m, i, a, stage, sn, co, wz);
    };
    links_fwd(m, body);
  }

  /* ---- the outward pass of the FUSE specialisations: pass 3 of stage s3 and pass 1 of stage s1 in ONE walk over the links
   * (-1: that half does not run).  A Runge-Kutta-Gill step is then
   *   P1(K1) P2(K1) [P3(K1) P1(K2)] P2(K2) [P3(K2) P1(K3)] P2(K3) [P3(K3) P1(K4)] P2(K4) [P3(K4) P1(REF)] P2(REF) P3(REF):
   * 11 passes and block barriers instead of 15, and pass 1 takes the new (sin, cos, q') of each joint from the registers
   * pass 3 has just computed them in.  At link i pass 3 reads U before pass 1 writes the new angular velocity into the same
   * slots; link i reads nothing of links > i.  Both halves sit in one function with one call site, selected by the
   * warp-uniform stages, so that the link body and the contact code exist once in the kernel (instruction cache); the
   * contacts of the tip run after the loop, when pass 3's carried values are dead. */
  RKFD_HD void outward(const ModelDev &m, int s3, int s1){
    const bool ref = s1 == ST_REF || s1 == ST_EVAL_REF;
    Acc a; acc_init(a);
    Kin kn; kin_init(kn);
    auto body = [&](const int i, auto Ktag){
      using Kt = decltype(Ktag);
      if( !Ctx::RIGID ) c.phase_sync(3);
      double sn = 0.0, co = 1.0, wz = 0.0;
      if( s3 >= 0 ) pass3_link<Kt>(m, i, a, s3, sn, co, wz);
      else if( JT<Kt>(i, m.link[i]) == J_REVOL ) revol_state(m, i, true, sn, co, wz);   /* first pass 1 of a step or evaluation */
      if( s1 >= 0 ) pass1_link<Kt>(m, i, kn, ref, sn, co, wz, false);
    };
    links_fwd(m, body);
    const int t = Spec::NL - 1; const LinkDev &L = m.link[t]; const int wx = Spec::wext_slot(t, L);
    if( s1 >= 0 && wx >= 0 ){ const V6 w = contacts(m, L, kn.Rw, kn.pw, kn.vl, kn.om, ref); st3(wx, w.l); st3(wx+3, w.a); }
  }


  /* =====================================================================================================
   * Rigid-contact solve of ONE environment, executed cooperatively by the lanes of its warp
   * (reference _rkFDSolverConstraint: rkfd_vert.c:327-336 / rkfd_mlcp.c:287-297).  `act` = lanes whose
   * environment has active rigid contacts; they are served one after the other, all lanes working on the
   * selected environment's scratch column:
   *   contact geometry + bias b      lanes over contacts        rkfd_vert.c:107-123
   *   A by 3N cached-ABA probes      lanes over probe columns   rkfd_vert.c:153-185, rkfd_util.c:163-181
   *   velocity bias / compensation   lanes over rows            rkfd_vert.c:189-232, rkfd_mlcp.c:146-188
   *   PGS (MLCP) or active-set QP    lanes over matrix columns  rkfd_mlcp.c:190-249, rkfd_opt_qp.c:43-181
   *   forces -> wrenches, friction state                        rkfd_vert.c:286-324, rkfd_mlcp.c:252-284
   * On the host harness a "warp" has one lane, which makes every loop sequential in the oracle's order.
   * ===================================================================================================== */
  RKFD_HD double &G(const ModelDev &m, int k, int i){ return c.W(m.ws_geo + GEO_DOUBLES*k + i); }
  RKFD_HD V3 g3(const ModelDev &m, int k, int i){ return v3(G(m,k,i), G(m,k,i+1), G(m,k,i+2)); }
  RKFD_HD void sg3(const ModelDev &m, int k, int i, V3 v){ G(m,k,i)=v.x; G(m,k,i+1)=v.y; G(m,k,i+2)=v.z; }
  RKFD_HD V3 w3(int o){ return v3(c.W(o), c.W(o+1), c.W(o+2)); }
  RKFD_HD void sw3(int o, V3 v){ c.W(o)=v.x; c.W(o+1)=v.y; c.W(o+2)=v.z; }

  /* one probe: unit force `axis` (world) at vertex `rl` (link frame) of link `Lc`; fills the increments of the
   * link accelerations da[col][link] ([EXT A-5] rkChainUpdateCachedABIPair: bias-only inward pass along the
   * path to the root with the cached articulated inertias, then the outward pass) */
  RKFD_HD void probe(const ModelDev &m, int col, int Lc, V3 rl, V3 axis, int Lb = -1, V3 vw = V3()){
    const int du0 = m.ws_du + col*6*m.nl, da0 = m.ws_da + col*6*m.nl;
    for(int k=0;k<6*m.nl;k++) c.W(du0+k) = 0.0;
    /* the unit force on the vertex's link and, when the partner moves, its opposite on the partner's link at the same world
     * point (rkfd_vert.c:166-175): two bias-only inward walks; the joint-space increments of links on both paths add up */
    for(int side=0; side<( Lb >= 0 ? 2 : 1 ); side++){
    V3 dpf, dpn; int i0 = Lc;
    if( side == 0 ){ const M3 Rw = ldm(m.link[Lc].frame_slot);
      const V3 fl = tmul(Rw, axis); dpf = -fl; dpn = -cross(rl, fl); }
    else { const int fb = m.link[Lb].frame_slot; const M3 RwB = ldm(fb);
      const V3 fl = tmul(RwB, axis), rb = tmul(RwB, vw - ld3(fb+9)); dpf = fl; dpn = cross(rb, fl); i0 = Lb; }
    for(int i=i0;;){
      const LinkDev &L = m.link[i]; const int sl = L.slot, ejt = eff_jt(L.jtype, sl);
      V3 paf = dpf, pan = dpn;
      switch(ejt){
      case J_REVOL: case J_PRISM: {
        const double du = ejt == J_REVOL ? -dpn.z : -dpf.z;
        c.W(du0+6*i) += du;
        const double k = Q(Spec::sc(i,L)+2)*du;
        paf = dpf + k*ld3(sl); pan = dpn + k*ld3(sl+3);
      } break;
      case J_SPHER: {
        const M3 E = tmm(ldm(sl+27), org_R(L));
        const V3 du = -tmul(E, dpn);
        sw3(du0+6*i, w3(du0+6*i) + du);
        const V3 k = mul(lds(sl+18), du);
        paf = dpf + mul(ldm(sl), k); pan = dpn + mul(ldm(sl+9), k);
      } break;
      case J_FLOAT: sw3(du0+6*i, w3(du0+6*i) + dpf); sw3(du0+6*i+3, w3(du0+6*i+3) + dpn); break;
      case J_CYLIN: case J_HOOKE: { double d2[2]; probe2_in(ejt, sl, dpf, dpn, d2, paf, pan); c.W(du0+6*i) += d2[0]; c.W(du0+6*i+1) += d2[1]; } break;
      default: break;
      }
      if( L.parent < 0 || ejt == J_FLOAT ) break;
      V3 vJ, wJ; const XF x = joint_xform<TagRT,false>(m, L, i, vJ, wJ);
      dpf = xf_mul(x, paf); dpn = xf_mul(x, pan) + cross(x.p, dpf);
      i = L.parent;
    }
    }
    for(int i=0;i<m.nl;i++){
      const LinkDev &L = m.link[i]; const int sl = L.slot, ejt = eff_jt(L.jtype, sl);
      V3 al = v3(0,0,0), aa = v3(0,0,0);
      if( L.parent >= 0 ){ al = w3(da0+6*L.parent); aa = w3(da0+6*L.parent+3); }
      V3 vJ, wJ; const XF x = joint_xform<TagRT,false>(m, L, i, vJ, wJ);
      V3 xl = xf_tmul(x, al + cross(aa, x.p)), xa = xf_tmul(x, aa);
      switch(ejt){
      case J_REVOL: case J_PRISM: {
        const double acc = Q(Spec::sc(i,L)+2)*( c.W(du0+6*i) - (dot(ld3(sl),xl) + dot(ld3(sl+3),xa)) );
        if( ejt == J_REVOL ) xa.z += acc; else xl.z += acc;
      } break;
      case J_SPHER: {
        const V3 rhs = w3(du0+6*i) - (tmul(ldm(sl), xl) + tmul(ldm(sl+9), xa));
        xa = xa + mul(tmm(ldm(sl+27), org_R(L)), mul(lds(sl+18), rhs));
      } break;
      case J_FLOAT: {   /* da = -IA^-1 dp */
        double iv[21], dp[6] = { c.W(du0+6*i), c.W(du0+6*i+1), c.W(du0+6*i+2), c.W(du0+6*i+3), c.W(du0+6*i+4), c.W(du0+6*i+5) }, r[6];
        for(int k=0;k<21;k++) iv[k] = c.S(sl+18+k);
        int k = 0;
        for(int a=0;a<6;a++) r[a] = 0;
        for(int a=0;a<6;a++) for(int b=a;b<6;b++){ r[a] -= iv[k]*dp[b]; if( b != a ) r[b] -= iv[k]*dp[a]; k++; }
        xl = v3(r[0],r[1],r[2]); xa = v3(r[3],r[4],r[5]);
      } break;
      case J_CYLIN: case J_HOOKE: { const double d2[2] = { c.W(du0+6*i), c.W(du0+6*i+1) }; probe2_out(ejt, sl, d2, xl, xa); } break;
      default: break;
      }
      sw3(da0+6*i, xl); sw3(da0+6*i+3, xa);
    }
  }

  /* =====================================================================================================
   * MLCP when every rigid contact of the environment sits on ONE link (an end effector on the floor, a free
   * body on the floor): the Delassus matrix factors as A = H Lambda H^T with the 6x6 inverse operational-space
   * inertia Lambda of that link and one 6-vector h = (axis, rho x axis) per contact row, so that
   *   - 6 cached-ABA probes (unit wrench components at the link origin) replace the 3N per-contact probes,
   *   - projected Gauss-Seidel runs on the 6-vector u = Lambda * (sum of contact wrenches): a row product is
   *     h.u and a force update adds g = Lambda h times the change - no N x N matrix exists,
   *   - the probes of up to 5 environments of the warp run at once (lanes over (environment, component)),
   *     the sweeps run one environment per lane.
   * Same equations as rkfd_mlcp.c:104-284 (including the row offsets of the friction sweep and the
   * unconditional commit of the friction type); sums are formed in a different order, so results agree with the
   * dense path to rounding.
   * ===================================================================================================== */
  RKFD_HD V3 w13(int o){ return v3(c.W1(o), c.W1(o+1), c.W1(o+2)); }
  RKFD_HD void sw13(int o, V3 v){ c.W1(o)=v.x; c.W1(o+1)=v.y; c.W1(o+2)=v.z; }

  /* acceleration response (link frame) of link Lc to the bias change (dpf, dpn) on itself ([EXT A-5]) */
  RKFD_HD void probe_link(const ModelDev &m, int Lc, V3 dpf, V3 dpn, V3 &ral, V3 &raa){
    double du[6*MAX_LINKS]; int pth[MAX_LINKS]; int np = 0;
    for(int i=Lc;;){
      const LinkDev &L = m.link[i]; const int sl = Spec::slot(i,L), jt = eff_jt(Spec::jtype(i,L), Spec::slot(i,L));
      pth[np] = i;
      V3 paf = dpf, pan = dpn;
      switch(jt){
      case J_REVOL: case J_PRISM: {
        const double d = jt == J_REVOL ? -dpn.z : -dpf.z;
        du[6*np] = d;
        const double k = Q(Spec::sc(i,L)+2)*d;
        paf = dpf + k*ld3(sl); pan = dpn + k*ld3(sl+3);
      } break;
      case J_SPHER: {
        const M3 E = tmm(ldm(sl+27), org_R(L));
        const V3 d = -tmul(E, dpn);
        du[6*np] = d.x; du[6*np+1] = d.y; du[6*np+2] = d.z;
        const V3 k = mul(lds(sl+18), d);
        paf = dpf + mul(ldm(sl), k); pan = dpn + mul(ldm(sl+9), k);
      } break;
      case J_FLOAT: du[6*np]=dpf.x; du[6*np+1]=dpf.y; du[6*np+2]=dpf.z; du[6*np+3]=dpn.x; du[6*np+4]=dpn.y; du[6*np+5]=dpn.z; break;
      case J_CYLIN: case J_HOOKE: { double d2[2]; probe2_in(jt, sl, dpf, dpn, d2, paf, pan); du[6*np] = d2[0]; du[6*np+1] = d2[1]; } break;
      default: break;
      }
      np++;
      if( Spec::parent(i,L) < 0 || jt == J_FLOAT ) break;
      V3 vJ, wJ; const XF x = joint_xform<TagRT,false>(m, L, i, vJ, wJ);
      dpf = xf_mul(x, paf); dpn = xf_mul(x, pan) + cross(x.p, dpf);
      i = Spec::parent(i,L);
    }
    V3 al = v3(0,0,0), aa = v3(0,0,0);
    for(int q=np-1;q>=0;q--){
      const int i = pth[q]; const LinkDev &L = m.link[i]; const int sl = Spec::slot(i,L), jt = eff_jt(Spec::jtype(i,L), Spec::slot(i,L));
      V3 vJ, wJ; const XF x = joint_xform<TagRT,false>(m, L, i, vJ, wJ);
      V3 xl = xf_tmul(x, al + cross(aa, x.p)), xa = xf_tmul(x, aa);
      switch(jt){
      case J_REVOL: case J_PRISM: {
        const double acc = Q(Spec::sc(i,L)+2)*( du[6*q] - (dot(ld3(sl),xl) + dot(ld3(sl+3),xa)) );
        if( jt == J_REVOL ) xa.z += acc; else xl.z += acc;
      } break;
      case J_SPHER: {
        const V3 rhs = v3(du[6*q],du[6*q+1],du[6*q+2]) - (tmul(ldm(sl), xl) + tmul(ldm(sl+9), xa));
        xa = xa + mul(tmm(ldm(sl+27), org_R(L)), mul(lds(sl+18), rhs));
      } break;
      case J_FLOAT: {   /* da = -IA^-1 dp */
        double r[6] = {0,0,0,0,0,0}; int k = 0;
        for(int a=0;a<6;a++) for(int b=a;b<6;b++){ const double iv = c.S(sl+18+k); r[a] -= iv*du[6*q+b]; if( b != a ) r[b] -= iv*du[6*q+a]; k++; }
        xl = v3(r[0],r[1],r[2]); xa = v3(r[3],r[4],r[5]);
      } break;
      case J_CYLIN: case J_HOOKE: { const double d2[2] = { du[6*q], du[6*q+1] }; probe2_out(jt, sl, d2, xl, xa); } break;
      default: break;
      }
      al = xl; aa = xa;
    }
    ral = al; raa = aa;
  }

  /* Lambda (6x6, column-major in W1[36 g ..]) of every contact-group link of every environment in `act`: lanes over
   * (environment of the warp with contacts, group, wrench component) */
  RKFD_HD void lambda_probes(const ModelDev &m, unsigned act){
    const int nlanes = c.lanes(), lane = c.lane();
    const int nact = RKFD_POPC64((unsigned long long)act), per = 6*m.nrg;
    for(int t=lane; t<per*nact; t+=nlanes){
      const int j = t/per, rem = t - per*j, g = rem/6, comp = rem - 6*g;
      const int Lc = m.rg_link[g]; const LinkDev &LL = m.link[Lc];
      const int fsl = Spec::frame_slot(Lc, LL);
      unsigned a = act; for(int q=0;q<j;q++) a &= a - 1;
      c.select(RKFD_FFS32(a) - 1);
      const M3 Rw = ldm(fsl);
      const int ax = comp < 3 ? comp : comp - 3;
      const V3 el = ax == 0 ? v3(Rw.xx, Rw.xy, Rw.xz) : ( ax == 1 ? v3(Rw.yx, Rw.yy, Rw.yz) : v3(Rw.zx, Rw.zy, Rw.zz) );   /* Rw^T e_ax */
      const V3 z = v3(0,0,0);
      V3 ral, raa;
      probe_link(m, Lc, comp < 3 ? -el : z, comp < 3 ? z : -el, ral, raa);
      sw13(36*g + 6*comp, mul(Rw, ral)); sw13(36*g + 6*comp+3, mul(Rw, raa));
      c.unselect();
    }
    c.gsync();
  }

  RKFD_HD void rigid_mlcp_single(const ModelDev &m, bool ref, unsigned act){
    lambda_probes(m, act);
    /* ---- one environment per lane from here on; the groups do not couple: projected Gauss-Seidel per group */
    if( RKFD_POPC64(cfl & m.rigid_mask) == 0 ) return;
    unsigned long long nfl = cfl;
    for(int g=0;g<m.nrg;g++) rigid_mlcp_group(m, ref, g, nfl);
    cfl = nfl;
  }
  RKFD_HD void rigid_mlcp_group(const ModelDev &m, bool ref, int g, unsigned long long &nfl){
    const int Lc = m.rg_link[g]; const LinkDev &LL = m.link[Lc];
    const int fsl = Spec::frame_slot(Lc, LL), wsl = Spec::wext_slot(Lc, LL);
    const unsigned long long fl = cfl;
    double lam[36];
#pragma unroll
    for(int i=0;i<36;i++) lam[i] = c.W1(36*g + i);     /* lam[6*col + row] */
    const M3 Rw = ldm(fsl); const V3 pw = ld3(fsl+9), vl = ld3(fsl+12), om = ld3(fsl+15);
    const V3 al = ld3(fsl+18), aa = ld3(fsl+21);
    const V3 vlw = mul(Rw, vl), omw = mul(Rw, om);
    /* contacts in (pair, vertex) order: geometry, rows h, responses g = Lambda h, bias b (rkfd_mlcp.c:104-188) */
    int N = 0;
    { int k = 0;
      for(int s=0;s<m.nslot;s++){
        if( !( (fl & m.rigid_mask) >> (2*s) & 1ull ) ) continue;
        const PairDev &pr = m.pair[m.slot_pair[s]]; const CellDev &cl = m.cell[pr.cell]; const BoxDev &bx = m.box[pr.box];
        if( cl.link != Lc ) continue;
        const int vi = cl.vofs + m.slot_vert[s];
        const V3 rl = v3(m.vert[3*vi], m.vert[3*vi+1], m.vert[3*vi+2]);
        const M3 Rb = box_R(bx); const V3 pb = v3(bx.p[0],bx.p[1],bx.p[2]);
        const V3 vw = pw + mul(Rw, rl), vb = tmul(Rb, vw - pb);
        V3 ax[3], prob;
        box_face(bx, Rb, vb, bx.half[0]-fabs(vb.x), bx.half[1]-fabs(vb.y), bx.half[2]-fabs(vb.z), ax[0], ax[1], ax[2], prob);
        const V3 refb = v3(c.gld(c.st.cref,3*s), c.gld(c.st.cref,3*s+1), c.gld(c.st.cref,3*s+2));
        const V3 d = vw - (pb + mul(Rb, refb));
        const V3 rho = vw - pw;
        V3 vel = vlw + cross(omw, rho);
        if( has_slide(pr) ) vel = vel + slide_vel(m, pr, Rw, pw, Rw, pw, vw, ax[0]);
        /* rkFDLinkPointWldAcc (rkfd_util.c:92-101): R ( a + alpha x r + w x (w x r) ) */
        const V3 r = tmul(Rw, rho);
        V3 accp = mul(Rw, al + cross(aa, r) + cross(om, cross(om, r)));
        if( grav_acc(m) ) accp.z -= GRAVITY;       /* link accelerations carry the fictitious base acceleration there */
        const double mu = ( (fl >> (2*s+1)) & 1ull ) ? pr.KF : pr.SF;
        const int o = W1_CT + W1_CTN*k;
        for(int i=0;i<3;i++){
          const V3 hl = ax[i], ha = cross(rho, ax[i]);
          const double h[6] = {hl.x, hl.y, hl.z, ha.x, ha.y, ha.z};
          double g[6], dg = 0;
#pragma unroll
          for(int rr=0;rr<6;rr++){ double sum = 0;
#pragma unroll
            for(int cc=0;cc<6;cc++) sum += lam[6*cc+rr]*h[cc];
            g[rr] = sum; }
#pragma unroll
          for(int rr=0;rr<6;rr++){ dg += h[rr]*g[rr]; c.W1(o+6*i+rr) = g[rr]; c.W1(o+18+6*i+rr) = h[rr]; }
          /* velocity level + compensation (rkfd_mlcp.c:146-188); relaxation on the diagonal */
          const double comp = pr.K * ( i == 0 ? 1.0 : mu ) * dot(d, ax[i]);
          c.W1(o+36+i) = dot(ax[i], accp)*m.dt + dot(vel, ax[i]) + comp;
          c.W1(o+39+i) = dg + pr.L;
          c.W1(o+42+i) = 0.0;
        }
        sw13(o+45, rho); sw13(o+48, prob); c.W1(o+51) = mu; c.W1(o+52) = (double)s;
        k++;
      }
      N = k; }
    if( N == 0 ) return;
    /* ---- projected Gauss-Seidel on u = Lambda * (sum of contact wrenches) (rkfd_mlcp.c:190-249) */
    double u[6] = {0,0,0,0,0,0};
    for(int cnt=0;cnt<m.max_iter;cnt++){
      for(int k=0;k<N;k++){
        const int o = W1_CT + W1_CTN*k; const double L = m.pair[m.slot_pair[(int)c.W1(o+52)]].L;
        double sum = 0;
#pragma unroll
        for(int rr=0;rr<6;rr++) sum += c.W1(o+18+rr)*u[rr];
        const double fo = c.W1(o+42), aoo = c.W1(o+39);
        sum += L*fo;
        double ff = -( c.W1(o+36) + sum - aoo*fo ) / aoo;
        ff = ff < ZTOL ? 0.0 : ff;
        const double dlt = ff - fo;
        c.W1(o+42) = ff;
#pragma unroll
        for(int rr=0;rr<6;rr++) u[rr] += c.W1(o+rr)*dlt;
      }
      for(int k=0;k<N;k++){
        const int o = W1_CT + W1_CTN*k; const double L = m.pair[m.slot_pair[(int)c.W1(o+52)]].L;
        double ff[2];
        for(int i=0;i<2;i++){           /* rows offset+0 / offset+1, as the reference reads them (:219-225) */
          const double aii = c.W1(o+39+i), fi = c.W1(o+42+i);
          double sum = 0;
#pragma unroll
          for(int rr=0;rr<6;rr++) sum += c.W1(o+18+6*i+rr)*u[rr];
          sum += L*fi;
          ff[i] = fabs(aii) < ZTOL ? 0.0 : -( c.W1(o+36+i) + sum - aii*fi ) / aii;
        }
        const double mu = c.W1(o+51), fn = c.W1(o+42);
        const double fnorm = ff[0]*ff[0] + ff[1]*ff[1];
        double fs = (mu*fn)*(mu*fn), f1, f2;
        if( fnorm < ZTOL || fs < ZTOL ){ f1 = 0.0; f2 = 0.0; }
        else if( fnorm > fs ){ fs /= fnorm; f1 = ff[0]*fs; f2 = ff[1]*fs; }
        else { f1 = ff[0]; f2 = ff[1]; }
        const double d1 = f1 - c.W1(o+43), d2 = f2 - c.W1(o+44);
        c.W1(o+43) = f1; c.W1(o+44) = f2;
#pragma unroll
        for(int rr=0;rr<6;rr++) u[rr] += c.W1(o+6+rr)*d1 + c.W1(o+12+rr)*d2;
      }
    }
    /* ---- f /= dt; forces, wrench on the link, friction state (rkfd_mlcp.c:252-284: committed regardless of
     * doUpRef, world components of f as "normal"/"tangential" - mirrored) */
    V3 wl = v3(0,0,0), wa = v3(0,0,0);
    for(int k=0;k<N;k++){
      const int o = W1_CT + W1_CTN*k; const int s = (int)c.W1(o+52);
      const V3 fw = (c.W1(o+42)/m.dt)*w13(o+18) + (c.W1(o+43)/m.dt)*w13(o+24) + (c.W1(o+44)/m.dt)*w13(o+30);
      const double mu = c.W1(o+51);
      const bool kin = sqrt(fw.y*fw.y + fw.z*fw.z) > mu*fw.x - ZTOL;
      if( kin ){ nfl |= 2ull << (2*s); const V3 prob = w13(o+48); c.gst(c.st.cref,3*s,prob.x); c.gst(c.st.cref,3*s+1,prob.y); c.gst(c.st.cref,3*s+2,prob.z); }
      else { nfl &= ~(2ull << (2*s)); slide_commit_static(m, s, Rw, pw, pw + w13(o+45), w13(o+18)); }
      /* rkFDContactForcePushWrench (rkfd_util.c:268-282) */
      const V3 pos = tmul(Rw, w13(o+45)), fll = tmul(Rw, fw);
      wl = wl + fll; wa = wa + cross(pos, fll);
      if( ref ){ c.gst(c.st.cf,3*s,fw.x); c.gst(c.st.cf,3*s+1,fw.y); c.gst(c.st.cf,3*s+2,fw.z); }
    }
    c.S(wsl) += wl.x; c.S(wsl+1) += wl.y; c.S(wsl+2) += wl.z;
    c.S(wsl+3) += wa.x; c.S(wsl+4) += wa.y; c.S(wsl+5) += wa.z;
  }

  /* =====================================================================================================
   * Vert (friction pyramid + least-squares QP by the active-set method, rkfd_vert.c:73-324, rkfd_opt_qp.c:43-181)
   * when every rigid contact sits on ONE link, one environment per lane, no N x N matrix:
   *   A = H Lambda H^T  (rows h = (axis, rho x axis), Lambda 6x6)  =>  Q = A^T A + diag(L) = diag(L) + H M H^T,
   *   M = Lambda^T (H^T H) Lambda,  c = A^T c0 = H w,  w = Lambda^T H^T c0.
   * The pyramid rows of a vertex only touch that vertex's 3 unknowns, so the equality-constrained problem of an
   * active-set iteration is solved exactly in closed form: with Pi_k the 3x3 projector onto the null space of the
   * active rows of vertex k and P = sum_k (1/L_k) H_k^T Pi_k H_k (6x6),
   *   (I + P M) v = -P w,   u = M v + w,   x*_k = -(1/L_k) Pi_k H_k u,
   * and the multipliers are the minimum-norm solutions of N_k^T l_k = (I - Pi_k) H_k u per vertex (1x1 / 2x2 / 3x3
   * systems) - the same x* and the same minimum-norm multipliers the reference takes from the pseudo-inverse of
   * the singular KKT matrix ([EXT A-14]), without a pseudo-inverse.  The active-set logic (identical-point test,
   * release of the most negative multipliers, step to the first blocking row, anti-cycling history) is the
   * reference's.
   * ===================================================================================================== */
  RKFD_HD bool solve6(double (&a)[36], double (&b)[6]){      /* a x = b by Gaussian elimination with partial pivoting; x -> b */
    for(int k=0;k<6;k++){
      int p = k; double big = fabs(a[6*k+k]);
      for(int i=k+1;i<6;i++) if( fabs(a[6*i+k]) > big ){ big = fabs(a[6*i+k]); p = i; }
      if( !(big > 0.0) ) return false;
      if( p != k ){ for(int j=0;j<6;j++){ const double t = a[6*k+j]; a[6*k+j] = a[6*p+j]; a[6*p+j] = t; } const double t = b[k]; b[k] = b[p]; b[p] = t; }
      const double inv = 1.0/a[6*k+k];
      for(int i=k+1;i<6;i++){ const double f = a[6*i+k]*inv; if( f != 0.0 ){ for(int j=k;j<6;j++) a[6*i+j] -= f*a[6*k+j]; b[i] -= f*b[k]; } }
    }
    for(int k=5;k>=0;k--){ double sum = b[k]; for(int j=k+1;j<6;j++) sum -= a[6*k+j]*b[j]; b[k] = sum/a[6*k+k]; }
    return true;
  }
  /* projector onto the null space of the active pyramid rows (mask am) of a vertex with friction coefficient fric */
  RKFD_HD void pyramid_projector(const ModelDev &m, unsigned am, double fric, double (&pi)[9]){
    const int na = RKFD_POPC64((unsigned long long)am);
    for(int i=0;i<9;i++) pi[i] = 0.0;
    if( na == 0 ){ pi[0] = pi[4] = pi[8] = 1.0; return; }
    if( na >= 3 ) return;
    const int i0 = RKFD_FFS32(am) - 1; const V3 a0 = v3(fric, m.sc_sin[i0], m.sc_cos[i0]);
    if( na == 1 ){
      const double inv = 1.0/dot(a0,a0);
      pi[0] = 1.0 - a0.x*a0.x*inv; pi[1] = -a0.x*a0.y*inv; pi[2] = -a0.x*a0.z*inv;
      pi[3] = pi[1]; pi[4] = 1.0 - a0.y*a0.y*inv; pi[5] = -a0.y*a0.z*inv;
      pi[6] = pi[2]; pi[7] = pi[5]; pi[8] = 1.0 - a0.z*a0.z*inv;
      return;
    }
    const int i1 = RKFD_FFS32(am & (am - 1)) - 1; const V3 a1 = v3(fric, m.sc_sin[i1], m.sc_cos[i1]);
    const V3 nn = cross(a0, a1); const double inv = 1.0/dot(nn,nn);
    pi[0] = nn.x*nn.x*inv; pi[1] = nn.x*nn.y*inv; pi[2] = nn.x*nn.z*inv;
    pi[3] = pi[1]; pi[4] = nn.y*nn.y*inv; pi[5] = nn.y*nn.z*inv;
    pi[6] = pi[2]; pi[7] = pi[5]; pi[8] = nn.z*nn.z*inv;
  }

  RKFD_HD void rigid_vert_single(const ModelDev &m, bool ref, unsigned act){
    /* contact groups (links in different chains) share ONE active-set iteration, as the reference's single QP does:
     * identical-point test, most negative multiplier, step length and history are global; the KKT solves decouple */
    lambda_probes(m, act);
    const unsigned long long fl = cfl;
    const int N = RKFD_POPC64(fl & m.rigid_mask);
    if( N == 0 ) return;
    const int pyr = m.pyramid, QP_MAXIT = 256;
    const int nrs = m.nmax/3, ohist = W1_CT + W1_CTN*nrs, hstr = qp_hist_stride(nrs), hw = (N + 2)/3;
    const int ng = m.nrg;
    /* contacts in (pair, vertex) order: rows h, compensated velocity-level bias c0 (rkfd_vert.c:107-123, 189-232);
     * per contact in W1: x (0..2) x* (3..5) h (18..35) c0 (36..38) fric (39) L (40) rho (45..47) prob (48..50) mu slot */
    { int k = 0;
      for(int s=0;s<m.nslot;s++){
        if( !( (fl & m.rigid_mask) >> (2*s) & 1ull ) ) continue;
        const PairDev &pr = m.pair[m.slot_pair[s]]; const CellDev &cl = m.cell[pr.cell]; const BoxDev &bx = m.box[pr.box];
        int g = 0; while( g < ng-1 && m.rg_link[g] != cl.link ) g++;
        const int fsl = Spec::frame_slot(cl.link, m.link[cl.link]);
        const M3 Rw = ldm(fsl); const V3 pw = ld3(fsl+9), vl = ld3(fsl+12), om = ld3(fsl+15);
        const V3 al = ld3(fsl+18), aa = ld3(fsl+21);
        const V3 vlw = mul(Rw, vl), omw = mul(Rw, om);
        const int vi = cl.vofs + m.slot_vert[s];
        const V3 rl = v3(m.vert[3*vi], m.vert[3*vi+1], m.vert[3*vi+2]);
        const M3 Rb = box_R(bx); const V3 pb = v3(bx.p[0],bx.p[1],bx.p[2]);
        const V3 vw = pw + mul(Rw, rl), vb = tmul(Rb, vw - pb);
        V3 ax[3], prob;
        box_face(bx, Rb, vb, bx.half[0]-fabs(vb.x), bx.half[1]-fabs(vb.y), bx.half[2]-fabs(vb.z), ax[0], ax[1], ax[2], prob);
        const V3 refb = v3(c.gld(c.st.cref,3*s), c.gld(c.st.cref,3*s+1), c.gld(c.st.cref,3*s+2));
        const V3 d = vw - (pb + mul(Rb, refb));
        const V3 rho = vw - pw;
        V3 vel = vlw + cross(omw, rho);
        if( has_slide(pr) ) vel = vel + slide_vel(m, pr, Rw, pw, Rw, pw, vw, ax[0]);
        const V3 r = tmul(Rw, rho);
        V3 accp = mul(Rw, al + cross(aa, r) + cross(om, cross(om, r)));
        if( grav_acc(m) ) accp.z -= GRAVITY;
        const double mu = ( (fl >> (2*s+1)) & 1ull ) ? pr.KF : pr.SF;
        const int o = W1_CT + W1_CTN*k;
        for(int i=0;i<3;i++){
          const V3 hl = ax[i], ha = cross(rho, ax[i]);
          const double h[6] = {hl.x, hl.y, hl.z, ha.x, ha.y, ha.z};
          const double c0 = dot(ax[i], accp)*m.dt + dot(vel, ax[i]) + pr.K * ( i == 0 ? 1.0 : mu ) * dot(d, ax[i]);
          for(int rr=0;rr<6;rr++) c.W1(o+18+6*i+rr) = h[rr];
          c.W1(o+36+i) = c0;
          c.W1(o+i) = i == 0 ? 1.0 : 0.0;            /* initial point f_n = 1 per vertex (rkfd_vert.c:234-244) */
        }
        c.W1(o+39) = mu*m.sc_cos[0]; c.W1(o+40) = pr.L; c.W1(o+41) = (double)g;
        sw13(o+45, rho); sw13(o+48, prob); c.W1(o+51) = mu; c.W1(o+52) = (double)s;
        k++;
      } }
    /* per group: M = Lambda^T G Lambda (row-major, written over Lambda in W1), w = Lambda^T hc   (Lambda[r][c] = lam[6c + r]) */
    double w[MAX_RG][6], u[MAX_RG][6];
    for(int g=0;g<ng;g++){
      double lam[36], G[36], hc[6], T[36];
      for(int i=0;i<36;i++){ lam[i] = c.W1(36*g + i); G[i] = 0.0; }
      for(int i=0;i<6;i++) hc[i] = 0.0;
      for(int k=0;k<N;k++){
        const int o = W1_CT + W1_CTN*k; if( (int)c.W1(o+41) != g ) continue;
        for(int i=0;i<3;i++){ const double c0 = c.W1(o+36+i);
          for(int rr=0;rr<6;rr++){ const double hr = c.W1(o+18+6*i+rr); hc[rr] += hr*c0; for(int cc=0;cc<6;cc++) G[6*rr+cc] += hr*c.W1(o+18+6*i+cc); } }
      }
      for(int r=0;r<6;r++) for(int cc=0;cc<6;cc++){ double sum = 0; for(int j=0;j<6;j++) sum += G[6*r+j]*lam[6*cc+j]; T[6*r+cc] = sum; }      /* G Lambda */
      for(int r=0;r<6;r++) for(int cc=0;cc<6;cc++){ double sum = 0; for(int j=0;j<6;j++) sum += lam[6*r+j]*T[6*j+cc]; c.W1(36*g + 6*r+cc) = sum; }   /* Lambda^T (G Lambda) */
      for(int r=0;r<6;r++){ double sum = 0; for(int j=0;j<6;j++) sum += lam[6*r+j]*hc[j]; w[g][r] = sum; }
    }
    /* initial active set (rkfd_opt_qp.c:27-40) */
    unsigned am[RIGID_MAX_SLOTS];
    for(int k=0;k<N;k++){
      const int o = W1_CT + W1_CTN*k; const double fric = c.W1(o+39); unsigned a = 0;
      for(int i=0;i<pyr;i++){ const double cond = fric*c.W1(o) + m.sc_sin[i]*c.W1(o+1) + m.sc_cos[i]*c.W1(o+2); if( fabs(cond) < ZTOL ) a |= 1u << i; }
      am[k] = a;
    }
    int nhist = 0;
    for(int iter=0; iter<QP_MAXIT; iter++){
      /* ---- x* of the equality-constrained problem, group by group */
      bool singular = false;
      for(int g=0;g<ng;g++){
      double P[36], M[36];
      for(int i=0;i<36;i++){ P[i] = 0.0; M[i] = c.W1(36*g + i); }
      for(int k=0;k<N;k++){
        const int o = W1_CT + W1_CTN*k; double pi[9];
        if( (int)c.W1(o+41) != g ) continue;
        pyramid_projector(m, am[k], c.W1(o+39), pi);
        const double il = 1.0/c.W1(o+40);
        for(int a=0;a<3;a++) for(int b=0;b<3;b++){
          const double pab = pi[3*a+b]*il; if( pab == 0.0 ) continue;
          for(int rr=0;rr<6;rr++){ const double ha = c.W1(o+18+6*a+rr)*pab; for(int cc=0;cc<6;cc++) P[6*rr+cc] += ha*c.W1(o+18+6*b+cc); }
        }
      }
      double K6[36], v[6];
      for(int r=0;r<6;r++){ double sum = 0; for(int cc=0;cc<6;cc++){ double pm = 0; for(int j=0;j<6;j++) pm += P[6*r+j]*M[6*j+cc]; K6[6*r+cc] = pm + (r == cc ? 1.0 : 0.0); sum += P[6*r+cc]*w[g][cc]; } v[r] = -sum; }
      if( !solve6(K6, v) ){ singular = true; break; }
      for(int r=0;r<6;r++){ double sum = w[g][r]; for(int j=0;j<6;j++) sum += M[6*r+j]*v[j]; u[g][r] = sum; }
      }
      if( singular ){ bad |= 2; break; }
      bool same = true, neg = false; double lmin = 0; bool first = true;
      for(int k=0;k<N;k++){
        const int o = W1_CT + W1_CTN*k; double pi[9]; const int gk = (int)c.W1(o+41);
        pyramid_projector(m, am[k], c.W1(o+39), pi);
        const double il = 1.0/c.W1(o+40);
        double hu[3];
        for(int a=0;a<3;a++){ double sum = 0; for(int rr=0;rr<6;rr++) sum += c.W1(o+18+6*a+rr)*u[gk][rr]; hu[a] = sum; }
        for(int a=0;a<3;a++){
          const double xs = -il*(pi[3*a]*hu[0] + pi[3*a+1]*hu[1] + pi[3*a+2]*hu[2]);
          c.W1(o+3+a) = xs;
          if( !(fabs(xs - c.W1(o+a)) < ZTOL) ) same = false;
        }
      }
      if( same ){
        /* multipliers: minimum-norm solution of N_k^T l_k = L_k x*_k + H_k u per vertex */
        for(int k=0;k<N;k++){
          const int o = W1_CT + W1_CTN*k; const unsigned a = am[k]; const int na = RKFD_POPC64((unsigned long long)a);
          c.W1(o) = c.W1(o+3); c.W1(o+1) = c.W1(o+4); c.W1(o+2) = c.W1(o+5);
          if( na == 0 ) continue;
          const double fric = c.W1(o+39), Lk = c.W1(o+40);
          V3 r;
          { const int gk = (int)c.W1(o+41);
            double hu[3]; for(int ax=0;ax<3;ax++){ double sum = 0; for(int rr=0;rr<6;rr++) sum += c.W1(o+18+6*ax+rr)*u[gk][rr]; hu[ax] = sum; }
            r = v3(Lk*c.W1(o+3) + hu[0], Lk*c.W1(o+4) + hu[1], Lk*c.W1(o+5) + hu[2]); }
          if( na == 1 ){
            const int i0 = RKFD_FFS32(a) - 1; const V3 a0 = v3(fric, m.sc_sin[i0], m.sc_cos[i0]);
            const double l = dot(a0, r)/dot(a0, a0);
            c.W1(o+6+0) = l;       /* multipliers of this vertex in slots 6.. (up to pyr <= 12 of them: 6..17) */
          } else if( na == 2 ){
            const int i0 = RKFD_FFS32(a) - 1, i1 = RKFD_FFS32(a & (a - 1)) - 1;
            const V3 a0 = v3(fric, m.sc_sin[i0], m.sc_cos[i0]), a1 = v3(fric, m.sc_sin[i1], m.sc_cos[i1]);
            const double g00 = dot(a0,a0), g01 = dot(a0,a1), g11 = dot(a1,a1), r0 = dot(a0,r), r1 = dot(a1,r);
            const double det = g00*g11 - g01*g01;
            c.W1(o+6+0) = (g11*r0 - g01*r1)/det; c.W1(o+6+1) = (g00*r1 - g01*r0)/det;
          } else {
            S3 sg; sg.xx=sg.xy=sg.xz=sg.yy=sg.yz=sg.zz=0;
            for(int i=0;i<pyr;i++) if( a >> i & 1u ){ const V3 ai = v3(fric, m.sc_sin[i], m.sc_cos[i]);
              sg.xx += ai.x*ai.x; sg.xy += ai.x*ai.y; sg.xz += ai.x*ai.z; sg.yy += ai.y*ai.y; sg.yz += ai.y*ai.z; sg.zz += ai.z*ai.z; }
            const V3 z = mul(sym3_inverse(sg), r);
            int t = 0;
            for(int i=0;i<pyr;i++) if( a >> i & 1u ){ c.W1(o+6+t) = fric*z.x + m.sc_sin[i]*z.y + m.sc_cos[i]*z.z; t++; }
          }
          for(int t=0;t<na;t++){ const double l = c.W1(o+6+t); if( l < 0 ) neg = true; if( first || l < lmin ){ lmin = l; first = false; } }
        }
        if( !neg ) break;                                  /* optimal */
        for(int k=0;k<N;k++){                               /* release every row within 1e-8 of the most negative multiplier (rkfd_opt_qp.c:117-131) */
          const int o = W1_CT + W1_CTN*k; unsigned a = am[k]; int t = 0;
          for(int i=0;i<pyr;i++) if( am[k] >> i & 1u ){ if( fabs(c.W1(o+6+t) - lmin) < 1.0e-8 ) a &= ~(1u << i); t++; }
          am[k] = a;
        }
        continue;
      }
      /* ---- step to the first blocking row, newly active rows (rkfd_opt_qp.c:133-151) */
      double alpha = 1.0;
      for(int k=0;k<N;k++){
        const int o = W1_CT + W1_CTN*k; const double fric = c.W1(o+39);
        const V3 x = w13(o), dx = w13(o+3) - x;
        for(int i=0;i<pyr;i++){
          if( am[k] >> i & 1u ) continue;
          const double ad = fric*dx.x + m.sc_sin[i]*dx.y + m.sc_cos[i]*dx.z;
          if( ad < 0 ){ const double cond = fric*x.x + m.sc_sin[i]*x.y + m.sc_cos[i]*x.z; const double t2 = (0.0 - cond)/ad; if( t2 < alpha ) alpha = t2; }
        }
      }
      double vv[MAX_RG][6], lx2 = 0;
      for(int g=0;g<ng;g++) for(int r=0;r<6;r++) vv[g][r] = 0.0;
      for(int k=0;k<N;k++){
        const int o = W1_CT + W1_CTN*k; const double fric = c.W1(o+39); const int gk = (int)c.W1(o+41);
        V3 x = w13(o); const V3 xs = w13(o+3);
        x = v3(x.x + alpha*(xs.x - x.x), x.y + alpha*(xs.y - x.y), x.z + alpha*(xs.z - x.z));
        sw13(o, x);
        for(int i=0;i<pyr;i++){
          if( am[k] >> i & 1u ) continue;
          const double cond = fric*x.x + m.sc_sin[i]*x.y + m.sc_cos[i]*x.z;
          if( fabs(cond) < ZTOL ) am[k] |= 1u << i;
        }
        lx2 += c.W1(o+40)*dot(x,x);
        for(int rr=0;rr<6;rr++) vv[gk][rr] += c.W1(o+18+rr)*x.x + c.W1(o+24+rr)*x.y + c.W1(o+30+rr)*x.z;
      }
      /* anti-cycling: same active set with the same objective value -> stop (rkfd_opt_qp.c:152-171) */
      double objv = 0.5*lx2;
      for(int g=0;g<ng;g++) for(int r=0;r<6;r++){ double sum = 0; for(int j=0;j<6;j++) sum += c.W1(36*g + 6*r+j)*vv[g][j]; objv += 0.5*vv[g][r]*sum + w[g][r]*vv[g][r]; }
      double pk[(RIGID_MAX_SLOTS + 2)/3];
      for(int k3=0;k3<hw;k3++){ double v = 0.0;
        for(int j=2;j>=0;j--){ const int k = 3*k3 + j; v = v*65536.0 + ( k < N ? (double)am[k] : 0.0 ); }
        pk[k3] = v; }
      bool endflag = false;
      for(int h=0;h<nhist && !endflag;h++){
        bool eq = true;
        for(int k3=0;k3<hw;k3++) if( pk[k3] != c.W1(ohist+h*hstr+k3) ){ eq = false; break; }
        if( eq && !(fabs(c.W1(ohist+h*hstr+hstr-1)/objv - 1.0) > 1.0e-8) ) endflag = true;
      }
      if( endflag ) break;
      if( nhist < QP_HIST ){
        for(int k3=0;k3<hw;k3++) c.W1(ohist+nhist*hstr+k3) = pk[k3];
        c.W1(ohist+nhist*hstr+hstr-1) = objv;
        nhist++;
      } else { bad |= 2; break; }
    }
    wk = 1u + 12u*(unsigned)((N < 5 ? N : 5) - 1) + (unsigned)(nhist < 11 ? nhist : 11);      /* contacts x iterations: the re-sort key */
    /* f = x / dt ; forces, wrench, friction state from the final active set (rkfd_vert.c:282, 286-324) */
    unsigned long long nfl = fl;
    for(int g=0;g<ng;g++){
    const int Lc = m.rg_link[g]; const LinkDev &LL = m.link[Lc];
    const int fsl = Spec::frame_slot(Lc, LL), wsl = Spec::wext_slot(Lc, LL);
    const M3 Rw = ldm(fsl);
    V3 wl = v3(0,0,0), wa = v3(0,0,0);
    for(int k=0;k<N;k++){
      const int o = W1_CT + W1_CTN*k; const int s = (int)c.W1(o+52);
      if( (int)c.W1(o+41) != g ) continue;
      const V3 fw = (c.W1(o)/m.dt)*w13(o+18) + (c.W1(o+1)/m.dt)*w13(o+24) + (c.W1(o+2)/m.dt)*w13(o+30);
      const bool flag = am[k] != 0;
      if( ref ){
        if( flag ){ nfl |= 2ull << (2*s); const V3 prob = w13(o+48); c.gst(c.st.cref,3*s,prob.x); c.gst(c.st.cref,3*s+1,prob.y); c.gst(c.st.cref,3*s+2,prob.z); }
        else { nfl &= ~(2ull << (2*s)); slide_commit_static(m, s, Rw, ld3(fsl+9), ld3(fsl+9) + w13(o+45), w13(o+18)); }
        c.gst(c.st.cf,3*s,fw.x); c.gst(c.st.cf,3*s+1,fw.y); c.gst(c.st.cf,3*s+2,fw.z);
      }
      const V3 pos = tmul(Rw, w13(o+45)), fll = tmul(Rw, fw);
      wl = wl + fll; wa = wa + cross(pos, fll);
    }
    c.S(wsl) += wl.x; c.S(wsl+1) += wl.y; c.S(wsl+2) += wl.z;
    c.S(wsl+3) += wa.x; c.S(wsl+4) += wa.y; c.S(wsl+5) += wa.z;
    }
    cfl = nfl;
  }

#include "rkfd_volume.cuh"

  RKFD_HD void rigid_solve(const ModelDev &m, bool ref, unsigned act){
    if constexpr ( Spec::NL == 0 ){ if( m.solver == S_VOLUME ){ rigid_volume(m, ref); return; } }
    if( m.rigid_link >= 0 ){ if( m.solver == S_MLCP ) rigid_mlcp_single(m, ref, act); else rigid_vert_single(m, ref, act); return; }
    const int nlanes = c.lanes(), lane = c.lane();
    while( act ){
      const int src = RKFD_FFS32(act) - 1; act &= act - 1;
      const unsigned long long fl = c.bcast(cfl, src);
      c.select(src);
      const int N = RKFD_POPC64(fl & m.rigid_mask), n = 3*N;
      const int ob = m.ws_b, of = m.ws_f, oA = m.ws_A;
      /* ---- contacts in (pair, vertex) order; geometry, bias acceleration b (rkfd_vert.c:107-123) */
      for(int k=lane;k<N;k+=nlanes){
        int s = 0, cnt = -1;
        for(;s<m.nslot;s++){ if( (fl & m.rigid_mask) >> (2*s) & 1ull ){ if( ++cnt == k ) break; } }
        const PairDev &pr = m.pair[m.slot_pair[s]]; const CellDev &cl = m.cell[pr.cell];
        const LinkDev &L = m.link[cl.link];
        const int vi = cl.vofs + m.slot_vert[s];
        const V3 rl = v3(m.vert[3*vi], m.vert[3*vi+1], m.vert[3*vi+2]);
        const M3 Rw = ldm(L.frame_slot); const V3 pw = ld3(L.frame_slot+9), vl = ld3(L.frame_slot+12), om = ld3(L.frame_slot+15);
        const V3 al = ld3(L.frame_slot+18), aa = ld3(L.frame_slot+21);
        const V3 vw = pw + mul(Rw, rl);
        /* the box: static, or carried by the partner link (its frame of this evaluation); rkFDChainPointRelativeVel / -Acc
         * (rkfd_util.c:42-60, 103-118): the vertex's link minus the partner's at the contact point, 0 for a static partner */
        BoxDev bx; M3 Rb; V3 pb, velB = v3(0,0,0), accB = v3(0,0,0); int Lb = -1;
        if( pr.mbox >= 0 ){
          const MBoxDev &mb = m.mbox[pr.mbox]; Lb = mb.link; const int fb = m.link[Lb].frame_slot;
          const M3 RwB = ldm(fb); const V3 pwB = ld3(fb+9), vlB = ld3(fb+12), omB = ld3(fb+15), alB = ld3(fb+18), aaB = ld3(fb+21);
          M3 Rl; Rl.xx=mb.R[0]; Rl.xy=mb.R[1]; Rl.xz=mb.R[2]; Rl.yx=mb.R[3]; Rl.yy=mb.R[4]; Rl.yz=mb.R[5]; Rl.zx=mb.R[6]; Rl.zy=mb.R[7]; Rl.zz=mb.R[8];
          Rb = mm(RwB, Rl); pb = pwB + mul(RwB, v3(mb.p[0], mb.p[1], mb.p[2]));
          for(int i=0;i<3;i++) bx.half[i] = mb.half[i];
          const V3 rB = tmul(RwB, vw - pwB);
          velB = mul(RwB, vlB) + cross(mul(RwB, omB), vw - pwB);
          accB = mul(RwB, alB + cross(aaB, rB) + cross(omB, cross(omB, rB)));
        } else { bx = m.box[pr.box]; Rb = box_R(bx); pb = v3(bx.p[0],bx.p[1],bx.p[2]); }
        const V3 vb = tmul(Rb, vw - pb);
        V3 nn, t1, t2, prob;
        box_face(bx, Rb, vb, bx.half[0]-fabs(vb.x), bx.half[1]-fabs(vb.y), bx.half[2]-fabs(vb.z), nn, t1, t2, prob);
        const V3 refb = v3(c.gld(c.st.cref,3*s), c.gld(c.st.cref,3*s+1), c.gld(c.st.cref,3*s+2));
        const V3 d = vw - (pb + mul(Rb, refb));
        V3 vel = mul(Rw, vl) + cross(mul(Rw, om), vw - pw) - velB;
        if( has_slide(pr) ){ const int fb = Lb >= 0 ? m.link[Lb].frame_slot : L.frame_slot;
          vel = vel + slide_vel(m, pr, Rw, pw, ldm(fb), ld3(fb+9), vw, nn); }
        /* rkFDLinkPointWldAcc (rkfd_util.c:92-101): R ( a + alpha x r + w x (w x r) ) */
        const V3 r = tmul(Rw, vw - pw);
        const V3 accp = mul(Rw, al + cross(aa, r) + cross(om, cross(om, r))) - accB;
        sg3(m,k,0,vw); sg3(m,k,3,nn); sg3(m,k,6,t1); sg3(m,k,9,t2); sg3(m,k,12,d); sg3(m,k,15,vel); sg3(m,k,18,prob); sg3(m,k,21,rl);
        G(m,k,24) = (double)s; G(m,k,25) = (double)cl.link; G(m,k,26) = (double)m.slot_pair[s]; G(m,k,27) = (double)Lb;
        c.W(ob+3*k) = dot(nn, accp); c.W(ob+3*k+1) = dot(t1, accp); c.W(ob+3*k+2) = dot(t2, accp);
      }
      c.gsync();
      /* ---- A: one probe per (contact, axis) column (rkfd_vert.c:153-185) */
      for(int col=lane;col<n;col+=nlanes){
        const int k = col/3, i = col - 3*k;
        probe(m, col, (int)G(m,k,25), g3(m,k,21), g3(m,k,3+3*i), (int)G(m,k,27), g3(m,k,0));
        const int da0 = m.ws_da + col*6*m.nl;
        for(int j=0;j<N;j++){
          const int Lj = (int)G(m,j,25), Bj = (int)G(m,j,27);
          const V3 dl = w3(da0+6*Lj), dal = w3(da0+6*Lj+3), r = g3(m,j,21);
          V3 resp = mul(ldm(m.link[Lj].frame_slot), dl + cross(dal, r));
          if( Bj >= 0 ){ const int fb = m.link[Bj].frame_slot; const M3 RwB = ldm(fb);
            const V3 rB = tmul(RwB, g3(m,j,0) - ld3(fb+9));
            resp = resp - mul(RwB, w3(da0+6*Bj) + cross(w3(da0+6*Bj+3), rB)); }
          c.W(oA+(3*j)*n+col) = dot(g3(m,j,3), resp); c.W(oA+(3*j+1)*n+col) = dot(g3(m,j,6), resp); c.W(oA+(3*j+2)*n+col) = dot(g3(m,j,9), resp);
        }
      }
      c.gsync();
      /* ---- velocity level: b <- b dt + axis . v_rel (rkfd_vert.c:189-206 / rkfd_mlcp.c:146-162) */
      for(int k=lane;k<N;k+=nlanes){
        const V3 vel = g3(m,k,15);
        c.W(ob+3*k)   = c.W(ob+3*k)  *m.dt + dot(vel, g3(m,k,3));
        c.W(ob+3*k+1) = c.W(ob+3*k+1)*m.dt + dot(vel, g3(m,k,6));
        c.W(ob+3*k+2) = c.W(ob+3*k+2)*m.dt + dot(vel, g3(m,k,9));
      }
      c.gsync();
      unsigned long long nfl = fl;
      if( m.solver == S_MLCP ){
        /* relaxation + compensation (rkfd_mlcp.c:164-188) */
        for(int k=lane;k<N;k+=nlanes){
          const PairDev &pr = m.pair[(int)G(m,k,26)]; const int s = (int)G(m,k,24); const V3 d = g3(m,k,12);
          const double mu = ( (fl >> (2*s+1)) & 1ull ) ? pr.KF : pr.SF;
          for(int i=0;i<3;i++) c.W(oA+(3*k+i)*n+3*k+i) += pr.L;
          c.W(ob+3*k)   += pr.K      * dot(d, g3(m,k,3));
          c.W(ob+3*k+1) += pr.K * mu * dot(d, g3(m,k,6));
          c.W(ob+3*k+2) += pr.K * mu * dot(d, g3(m,k,9));
        }
        for(int i=lane;i<n;i+=nlanes) c.W(of+i) = 0.0;
        c.gsync();
        /* projected Gauss-Seidel (rkfd_mlcp.c:190-249); the friction sweep reads rows offset+0 / offset+1 as the
         * reference does (:219-225) */
        for(int cnt=0;cnt<m.max_iter;cnt++){
          for(int k=0;k<N;k++){
            const int o = 3*k; double part = 0;
            for(int j=lane;j<n;j+=nlanes) part += c.W(oA+o*n+j)*c.W(of+j);
            const double sum = c.allsum(part), aoo = c.W(oA+o*n+o);
            const double ff = -( c.W(ob+o) + sum - aoo*c.W(of+o) ) / aoo;
            c.gsync();
            if( lane == 0 ) c.W(of+o) = ff < ZTOL ? 0.0 : ff;
            c.gsync();
          }
          for(int k=0;k<N;k++){
            const int o = 3*k; double ff[2];
            for(int i=0;i<2;i++){
              const double aii = c.W(oA+(o+i)*n+o+i);
              double part = 0;
              for(int j=lane;j<n;j+=nlanes) part += c.W(oA+(o+i)*n+j)*c.W(of+j);
              const double sum = c.allsum(part);
              ff[i] = fabs(aii) < ZTOL ? 0.0 : -( c.W(ob+o+i) + sum - aii*c.W(of+o+i) ) / aii;
            }
            const PairDev &pr = m.pair[(int)G(m,k,26)]; const int s = (int)G(m,k,24);
            const double mu = ( (fl >> (2*s+1)) & 1ull ) ? pr.KF : pr.SF;
            const double fnorm = ff[0]*ff[0] + ff[1]*ff[1];
            double fs = (mu*c.W(of+o))*(mu*c.W(of+o)), f1, f2;
            if( fnorm < ZTOL || fs < ZTOL ){ f1 = 0.0; f2 = 0.0; }
            else if( fnorm > fs ){ fs /= fnorm; f1 = ff[0]*fs; f2 = ff[1]*fs; }
            else { f1 = ff[0]; f2 = ff[1]; }
            c.gsync();
            if( lane == 0 ){ c.W(of+o+1) = f1; c.W(of+o+2) = f2; }
            c.gsync();
          }
        }
        /* f /= dt; forces, wrenches, friction state (rkfd_mlcp.c:252-284: committed regardless of doUpRef,
         * world components of f as "normal"/"tangential" - mirrored) */
        for(int k=0;k<N;k++){
          const int s = (int)G(m,k,24); const PairDev &pr = m.pair[(int)G(m,k,26)];
          const V3 fw = (c.W(of+3*k)/m.dt)*g3(m,k,3) + (c.W(of+3*k+1)/m.dt)*g3(m,k,6) + (c.W(of+3*k+2)/m.dt)*g3(m,k,9);
          const double mu = ( (fl >> (2*s+1)) & 1ull ) ? pr.KF : pr.SF;
          const bool kin = sqrt(fw.y*fw.y + fw.z*fw.z) > mu*fw.x - ZTOL;
          if( kin ) nfl |= 2ull << (2*s); else nfl &= ~(2ull << (2*s));
          if( lane == 0 ){
            push_rigid(m, k, fw, ref);
            if( kin ){ const V3 prob = g3(m,k,18); c.gst(c.st.cref,3*s,prob.x); c.gst(c.st.cref,3*s+1,prob.y); c.gst(c.st.cref,3*s+2,prob.z); }
            else slide_commit_dense(m, k);
          }
        }
      } else {
        nfl = qp_vert(m, ref, fl, N);
      }
      c.gsync();
      c.unselect();
      if( lane == src ) cfl = nfl;
    }
  }

  /* rkFDContactForcePushWrench (rkfd_util.c:268-282) for rigid contact k of the selected environment */
  RKFD_HD void push_rigid(const ModelDev &m, int k, V3 fw, bool ref){
    const LinkDev &L = m.link[(int)G(m,k,25)]; const int s = (int)G(m,k,24);
    const M3 Rw = ldm(L.frame_slot); const V3 pw = ld3(L.frame_slot+9);
    const V3 pos = tmul(Rw, g3(m,k,0) - pw), fl = tmul(Rw, fw);
    const V3 t = cross(pos, fl);
    c.S(L.wext_slot) += fl.x; c.S(L.wext_slot+1) += fl.y; c.S(L.wext_slot+2) += fl.z;
    c.S(L.wext_slot+3) += t.x; c.S(L.wext_slot+4) += t.y; c.S(L.wext_slot+5) += t.z;
    const int Lb = (int)G(m,k,27);
    if( Lb >= 0 ){          /* the partner takes the opposite force at the same point (rkfd_util.c:276-278) */
      const LinkDev &B = m.link[Lb]; const M3 RwB = ldm(B.frame_slot);
      const V3 posB = tmul(RwB, g3(m,k,0) - ld3(B.frame_slot+9)), flB = tmul(RwB, v3(-fw.x, -fw.y, -fw.z)), tB = cross(posB, flB);
      c.S(B.wext_slot) += flB.x; c.S(B.wext_slot+1) += flB.y; c.S(B.wext_slot+2) += flB.z;
      c.S(B.wext_slot+3) += tB.x; c.S(B.wext_slot+4) += tB.y; c.S(B.wext_slot+5) += tB.z;
    }
    if( ref ){ c.gst(c.st.cf,3*s,fw.x); c.gst(c.st.cf,3*s+1,fw.y); c.gst(c.st.cf,3*s+2,fw.z); }
  }

  /* a rigid contact committed as sticking: its anchor rides on the belts of the pair (rkFDUpdateRefSlide, rkfd_mlcp.c:279,
   * rkfd_vert.c:318).  Static partner, vertex link frame (Rw, pw): the single-link paths */
  RKFD_HD void slide_commit_static(const ModelDev &m, int s, const M3 &Rw, V3 pw, V3 vw, V3 n){
    const PairDev &pr = m.pair[m.slot_pair[s]];
    if( !has_slide(pr) ) return;
    const BoxDev &bx = m.box[pr.box];
    const V3 db = slide_ref_shift(m, pr, Rw, pw, box_lR(bx), v3(0,0,0), box_R(bx), vw, n);
    c.gst(c.st.cref,3*s, c.gld(c.st.cref,3*s) + db.x); c.gst(c.st.cref,3*s+1, c.gld(c.st.cref,3*s+1) + db.y); c.gst(c.st.cref,3*s+2, c.gld(c.st.cref,3*s+2) + db.z);
  }
  /* the same for rigid contact k of the dense path (geometry record G; the partner may move) */
  RKFD_HD void slide_commit_dense(const ModelDev &m, int k){
    const PairDev &pr = m.pair[(int)G(m,k,26)];
    if( !has_slide(pr) ) return;
    const int s = (int)G(m,k,24), Lv = (int)G(m,k,25), Lb = (int)G(m,k,27);
    const int fv = m.link[Lv].frame_slot; const M3 Rw = ldm(fv); const V3 pw = ld3(fv+9);
    M3 Rpl, Rbw; V3 pp = v3(0,0,0);
    if( Lb >= 0 ){ const MBoxDev &mb = m.mbox[pr.mbox]; const int fb = m.link[Lb].frame_slot; Rpl = ldm(fb); pp = ld3(fb+9);
      M3 Rl; Rl.xx=mb.R[0]; Rl.xy=mb.R[1]; Rl.xz=mb.R[2]; Rl.yx=mb.R[3]; Rl.yy=mb.R[4]; Rl.yz=mb.R[5]; Rl.zx=mb.R[6]; Rl.zy=mb.R[7]; Rl.zz=mb.R[8];
      Rbw = mm(Rpl, Rl); }
    else { const BoxDev &bx = m.box[pr.box]; Rpl = box_lR(bx); Rbw = box_R(bx); }
    const V3 db = slide_ref_shift(m, pr, Rw, pw, Rpl, pp, Rbw, g3(m,k,0), g3(m,k,3));
    c.gst(c.st.cref,3*s, c.gld(c.st.cref,3*s) + db.x); c.gst(c.st.cref,3*s+1, c.gld(c.st.cref,3*s+1) + db.y); c.gst(c.st.cref,3*s+2, c.gld(c.st.cref,3*s+2) + db.z);
  }

  /* Vert: friction pyramid + least-squares QP by the active-set method (rkfd_vert.c:73-103, 208-324;
   * rkFDQPSolveASM rkfd_opt_qp.c:43-181).  The KKT system [[-Q, Aw^T],[Aw, 0]] [x; l] = [c; 0] of every
   * iteration is solved through its Schur complement S = Aw Q^-1 Aw^T: l = S^+ (Aw Q^-1 c) (pseudo-inverse of
   * the small PSD matrix by cyclic Jacobi), x = Q^-1 (Aw^T l - c), which is the minimum-norm solution the
   * reference obtains from zLESolveMP on the full KKT matrix ([EXT A-14]; redundant active rows only make
   * the multipliers non-unique).  Returns the new contact flags of the selected environment. */
  RKFD_HD unsigned long long qp_vert(const ModelDev &m, bool ref, unsigned long long fl, int N){
    const int nlanes = c.lanes(), lane = c.lane();
    const int n = 3*N, pyr = m.pyramid, mc = pyr*N;
    const int nx = m.nmax, mx = m.pyramid*(m.nmax/3);
    const int ob = m.ws_b, of = m.ws_f, oA = m.ws_A;
    int o = m.ws_qp;
    const int oQ = o; o += nx*nx; const int oQi = o; o += nx*nx; const int oc = o; o += nx; const int og = o; o += nx;
    const int ox = o; o += nx; const int oxs = o; o += nx; const int onf = o; o += 3*mx; const int oidx = o; o += mx;
    const int oY = o; o += nx*mx; const int oS = o; o += mx*mx; const int oV = o; o += mx*mx; const int olam = o; o += mx;
    const int orhs = o; o += mx; const int oact = o; o += mx; const int ohist = o;     /* history: QP_HIST x (mx+1) */
    const int QP_HIST = 32, QP_MAXIT = 256;
    /* pyramid rows and compensated bias c (rkfd_vert.c:73-103, 208-232) */
    for(int k=lane;k<N;k+=nlanes){
      const PairDev &pr = m.pair[(int)G(m,k,26)]; const int sidx = (int)G(m,k,24); const V3 d = g3(m,k,12);
      const double mu = ( (fl >> (2*sidx+1)) & 1ull ) ? pr.KF : pr.SF;
      const double fric = mu*m.sc_cos[0];
      for(int i=0;i<pyr;i++){ c.W(onf+3*(pyr*k+i)) = fric; c.W(onf+3*(pyr*k+i)+1) = m.sc_sin[i]; c.W(onf+3*(pyr*k+i)+2) = m.sc_cos[i]; }
      c.W(of+3*k)   = c.W(ob+3*k)   + pr.K      * dot(d, g3(m,k,3));
      c.W(of+3*k+1) = c.W(ob+3*k+1) + pr.K * mu * dot(d, g3(m,k,6));
      c.W(of+3*k+2) = c.W(ob+3*k+2) + pr.K * mu * dot(d, g3(m,k,9));
    }
    c.gsync();
    /* Q = A^T A + L, c <- A^T c (rkfd_vert.c:267-279) */
    for(int e=lane;e<n*n;e+=nlanes){
      const int i = e/n, j = e - i*n; double sum = 0;
      for(int k=0;k<n;k++) sum += c.W(oA+k*n+i)*c.W(oA+k*n+j);
      if( i == j ) sum += m.pair[(int)G(m,i/3,26)].L;
      c.W(oQ+e) = sum; c.W(oQi+e) = (i == j) ? 1.0 : 0.0;
    }
    for(int i=lane;i<n;i+=nlanes){ double sum = 0; for(int j=0;j<n;j++) sum += c.W(oA+j*n+i)*c.W(of+j); c.W(oc+i) = sum; }
    c.gsync();
    /* Q^-1 by Gauss-Jordan on [Q | I] (Q is symmetric positive definite); the copy of Q is consumed */
    for(int e=lane;e<n*n;e+=nlanes) c.W(oY+e) = c.W(oQ+e);
    c.gsync();
    for(int k=0;k<n;k++){
      const double piv = 1.0/c.W(oY+k*n+k);
      c.gsync();
      for(int j=lane;j<n;j+=nlanes){ c.W(oY+k*n+j) *= piv; c.W(oQi+k*n+j) *= piv; }
      c.gsync();
      for(int e=lane;e<n*n;e+=nlanes){
        const int i = e/n, j = e - i*n;
        if( i == k ) continue;
        const double fac = c.W(oY+i*n+k);
        if( j != k ) c.W(oY+i*n+j) -= fac*c.W(oY+k*n+j);
        c.W(oQi+i*n+j) -= fac*c.W(oQi+k*n+j);
      }
      c.gsync();
      for(int i=lane;i<n;i+=nlanes) if( i != k ) c.W(oY+i*n+k) = 0.0;
      c.gsync();
    }
    /* g = Q^-1 c ; initial point f_n = 1 per vertex (rkfd_vert.c:234-244); initial active set (rkfd_opt_qp.c:27-40) */
    for(int i=lane;i<n;i+=nlanes){ double sum = 0; for(int j=0;j<n;j++) sum += c.W(oQi+i*n+j)*c.W(oc+j); c.W(og+i) = sum; c.W(ox+i) = (i%3 == 0) ? 1.0 : 0.0; }
    c.gsync();
    for(int r=lane;r<mc;r+=nlanes){
      const int k = r/pyr;
      const double cond = c.W(onf+3*r)*c.W(ox+3*k) + c.W(onf+3*r+1)*c.W(ox+3*k+1) + c.W(onf+3*r+2)*c.W(ox+3*k+2);
      c.W(oidx+r) = fabs(cond) < ZTOL ? 1.0 : 0.0;
    }
    c.gsync();
    int nhist = 0;
    for(int iter=0; iter<QP_MAXIT; iter++){
      /* active list in ascending order */
      int ma = 0;
      for(int r=0;r<mc;r++) if( c.W(oidx+r) != 0.0 ){ if( lane == 0 ) c.W(oact+ma) = (double)r; ma++; }
      c.gsync();
      /* Y_t = Q^-1 nf_t^T ; rhs_t = nf_t . g ; S = Aw Y */
      for(int e=lane;e<ma*n;e+=nlanes){
        const int t = e/n, i = e - t*n, r = (int)c.W(oact+t), k = r/pyr;
        c.W(oY+t*n+i) = c.W(oQi+i*n+3*k)*c.W(onf+3*r) + c.W(oQi+i*n+3*k+1)*c.W(onf+3*r+1) + c.W(oQi+i*n+3*k+2)*c.W(onf+3*r+2);
      }
      for(int t=lane;t<ma;t+=nlanes){ const int r = (int)c.W(oact+t), k = r/pyr;
        c.W(orhs+t) = c.W(onf+3*r)*c.W(og+3*k) + c.W(onf+3*r+1)*c.W(og+3*k+1) + c.W(onf+3*r+2)*c.W(og+3*k+2); }
      c.gsync();
      for(int e=lane;e<ma*ma;e+=nlanes){
        const int t = e/ma, u = e - t*ma, r = (int)c.W(oact+t), k = r/pyr;
        c.W(oS+e) = c.W(onf+3*r)*c.W(oY+u*n+3*k) + c.W(onf+3*r+1)*c.W(oY+u*n+3*k+1) + c.W(onf+3*r+2)*c.W(oY+u*n+3*k+2);
        c.W(oV+e) = (t == u) ? 1.0 : 0.0;
      }
      c.gsync();
      /* l = S^+ rhs: Jacobi eigen-decomposition of the symmetric S (ma x ma) in the PARALLEL (round-robin) ordering:
       * a sweep is me-1 rounds of me/2 rotations on disjoint index pairs (me = ma rounded up to even); the lanes
       * first compute the rotations of the round, then apply all of them to the columns of S and V, then to the
       * rows of S - three warp barriers per round instead of three per rotation (ma = 24: 69 instead of 828 per
       * sweep), and every lane has work.  (cs, sn) of the round live behind the anti-cycling history. */
      { const int me = (ma + 1) & ~1, np = me/2, ocs = ohist + QP_HIST*(mx+1);
        for(int sweep=0; sweep<40 && ma>1; sweep++){
          double part = 0;
          for(int e=lane;e<ma*ma;e+=nlanes){ const int t = e/ma, u = e - t*ma; if( u > t ) part += c.W(oS+e)*c.W(oS+e); }
          const double off = c.allsum(part);
          if( off < 1.0e-300 ) break;
          for(int rnd=0; rnd<me-1; rnd++){
            /* pair i of the round: (me-1, rnd) for i = 0, ((rnd+i) mod (me-1), (rnd+me-1-i) mod (me-1)) otherwise */
            for(int i=lane;i<np;i+=nlanes){
              int p = i == 0 ? me-1 : (rnd + i) % (me-1), q = i == 0 ? rnd : (rnd + me-1 - i) % (me-1);
              if( p > q ){ const int t = p; p = q; q = t; }
              double cs = 1.0, sn = 0.0;
              if( q < ma ){
                const double apq = c.W(oS+p*ma+q);
                if( !(fabs(apq) < 1.0e-300) ){
                  const double th = (c.W(oS+q*ma+q) - c.W(oS+p*ma+p))/(2.0*apq);
                  const double tt = (th >= 0 ? 1.0 : -1.0)/(fabs(th) + sqrt(th*th + 1.0));
                  cs = 1.0/sqrt(tt*tt + 1.0); sn = tt*cs;
                }
              }
              c.W(ocs+2*i) = cs; c.W(ocs+2*i+1) = sn;
            }
            c.gsync();
            for(int e=lane;e<np*ma;e+=nlanes){          /* columns p, q of S and V */
              const int i = e/ma, k = e - i*ma;
              int p = i == 0 ? me-1 : (rnd + i) % (me-1), q = i == 0 ? rnd : (rnd + me-1 - i) % (me-1);
              if( p > q ){ const int t = p; p = q; q = t; }
              if( q >= ma ) continue;
              const double cs = c.W(ocs+2*i), sn = c.W(ocs+2*i+1);
              const double akp = c.W(oS+k*ma+p), akq = c.W(oS+k*ma+q); c.W(oS+k*ma+p) = cs*akp - sn*akq; c.W(oS+k*ma+q) = sn*akp + cs*akq;
              const double vkp = c.W(oV+k*ma+p), vkq = c.W(oV+k*ma+q); c.W(oV+k*ma+p) = cs*vkp - sn*vkq; c.W(oV+k*ma+q) = sn*vkp + cs*vkq;
            }
            c.gsync();
            for(int e=lane;e<np*ma;e+=nlanes){          /* rows p, q of S */
              const int i = e/ma, k = e - i*ma;
              int p = i == 0 ? me-1 : (rnd + i) % (me-1), q = i == 0 ? rnd : (rnd + me-1 - i) % (me-1);
              if( p > q ){ const int t = p; p = q; q = t; }
              if( q >= ma ) continue;
              const double cs = c.W(ocs+2*i), sn = c.W(ocs+2*i+1);
              const double apk = c.W(oS+p*ma+k), aqk = c.W(oS+q*ma+k); c.W(oS+p*ma+k) = cs*apk - sn*aqk; c.W(oS+q*ma+k) = sn*apk + cs*aqk;
            }
            c.gsync();
          }
        }
      }
      double lmax = 0;
      for(int t=0;t<ma;t++) lmax = fmax(lmax, fabs(c.W(oS+t*ma+t)));
      for(int t=lane;t<ma;t+=nlanes){
        double sum = 0;
        for(int e=0;e<ma;e++){
          const double ev = c.W(oS+e*ma+e);
          if( fabs(ev) <= 1.0e-11*lmax ) continue;
          double pr = 0; for(int u=0;u<ma;u++) pr += c.W(oV+u*ma+e)*c.W(orhs+u);
          sum += c.W(oV+t*ma+e)*pr/ev;
        }
        c.W(olam+t) = sum;
      }
      c.gsync();
      /* x* = sum_t l_t Y_t - g */
      for(int i=lane;i<n;i+=nlanes){ double sum = -c.W(og+i); for(int t=0;t<ma;t++) sum += c.W(olam+t)*c.W(oY+t*n+i); c.W(oxs+i) = sum; }
      c.gsync();
      bool same = true;
      for(int i=0;i<n;i++) if( !(fabs(c.W(oxs+i) - c.W(ox+i)) < ZTOL) ){ same = false; break; }
#ifdef RKFD_QP_DEBUG
      { double mincond = 1e300, maxres = 0; for(int r=0;r<mc;r++){ const int k=r/pyr; const double cd = c.W(onf+3*r)*c.W(ox+3*k)+c.W(onf+3*r+1)*c.W(ox+3*k+1)+c.W(onf+3*r+2)*c.W(ox+3*k+2); if(cd<mincond) mincond=cd; }
        for(int t=0;t<ma;t++){ const int r=(int)c.W(oact+t), k=r/pyr; const double cd = c.W(onf+3*r)*c.W(oxs+3*k)+c.W(onf+3*r+1)*c.W(oxs+3*k+1)+c.W(onf+3*r+2)*c.W(oxs+3*k+2); if(fabs(cd)>maxres) maxres=fabs(cd); }
        double lmn=1e300; for(int t=0;t<ma;t++) if(c.W(olam+t)<lmn) lmn=c.W(olam+t);
        printf("iter %d ma %d same %d mincond(x) %.3e  |Aw x*| %.3e  lmin %.3e lmax_eig %.3e\n", iter, ma, (int)same, mincond, maxres, lmn, lmax); }
#endif
      if( same ){
        c.gsync();
        for(int i=lane;i<n;i+=nlanes) c.W(ox+i) = c.W(oxs+i);
        bool neg = false; double lmin = 0;
        for(int t=0;t<ma;t++){ const double l = c.W(olam+t); if( l < 0 ) neg = true; if( t == 0 || l < lmin ) lmin = l; }
        if( !neg ){ c.gsync(); break; }                                  /* optimal */
        c.gsync();
        for(int t=lane;t<ma;t+=nlanes) if( fabs(c.W(olam+t) - lmin) < 1.0e-8 ) c.W(oidx+(int)c.W(oact+t)) = 0.0;
        c.gsync();
        continue;
      }
      /* STEP2: step length to the first blocking constraint, new active constraints (rkfd_opt_qp.c:133-151) */
      double alpha = 1.0;
      for(int r=0;r<mc;r++){
        if( c.W(oidx+r) != 0.0 ) continue;
        const int k = r/pyr;
        const double ad = c.W(onf+3*r)*(c.W(oxs+3*k)-c.W(ox+3*k)) + c.W(onf+3*r+1)*(c.W(oxs+3*k+1)-c.W(ox+3*k+1)) + c.W(onf+3*r+2)*(c.W(oxs+3*k+2)-c.W(ox+3*k+2));
        if( ad < 0 ){
          const double cond = c.W(onf+3*r)*c.W(ox+3*k) + c.W(onf+3*r+1)*c.W(ox+3*k+1) + c.W(onf+3*r+2)*c.W(ox+3*k+2);
          const double t2 = (0.0 - cond)/ad; if( t2 < alpha ) alpha = t2;
        }
      }
      c.gsync();
      for(int i=lane;i<n;i+=nlanes) c.W(ox+i) += alpha*(c.W(oxs+i) - c.W(ox+i));
      c.gsync();
      for(int r=lane;r<mc;r+=nlanes){
        if( c.W(oidx+r) != 0.0 ) continue;
        const int k = r/pyr;
        const double cond = c.W(onf+3*r)*c.W(ox+3*k) + c.W(onf+3*r+1)*c.W(ox+3*k+1) + c.W(onf+3*r+2)*c.W(ox+3*k+2);
        if( fabs(cond) < ZTOL ) c.W(oidx+r) = 1.0;
      }
      c.gsync();
      /* anti-cycling: same active set with the same objective value -> stop (rkfd_opt_qp.c:152-171) */
      double objv = 0;
      for(int i=0;i<n;i++){ double sum = 0; for(int j=0;j<n;j++) sum += c.W(oQ+i*n+j)*c.W(ox+j); objv += 0.5*c.W(ox+i)*sum + c.W(oc+i)*c.W(ox+i); }
      bool endflag = false;
      for(int h=0;h<nhist && !endflag;h++){
        bool eq = true;
        for(int r=0;r<mc;r++) if( c.W(oidx+r) != c.W(ohist+h*(mx+1)+r) ){ eq = false; break; }
        if( eq && !(fabs(c.W(ohist+h*(mx+1)+mx)/objv - 1.0) > 1.0e-8) ) endflag = true;
      }
      if( endflag ) break;
      if( nhist < QP_HIST ){
        c.gsync();
        for(int r=lane;r<mc;r+=nlanes) c.W(ohist+nhist*(mx+1)+r) = c.W(oidx+r);
        if( lane == 0 ) c.W(ohist+nhist*(mx+1)+mx) = objv;
        nhist++;
        c.gsync();
      } else { bad |= 2; break; }
    }
    /* f = x / dt ; forces, wrenches, friction state from the final active set (rkfd_vert.c:282, 286-324) */
    unsigned long long nfl = fl;
    for(int k=0;k<N;k++){
      const int sidx = (int)G(m,k,24);
      const V3 fw = (c.W(ox+3*k)/m.dt)*g3(m,k,3) + (c.W(ox+3*k+1)/m.dt)*g3(m,k,6) + (c.W(ox+3*k+2)/m.dt)*g3(m,k,9);
      bool flag = false;
      for(int i=0;i<pyr;i++) if( c.W(oidx+pyr*k+i) != 0.0 ){ flag = true; break; }
      if( ref ){ if( flag ) nfl |= 2ull << (2*sidx); else nfl &= ~(2ull << (2*sidx)); }
      if( lane == 0 ){
        push_rigid(m, k, fw, ref);
        if( ref && flag ){ const V3 prob = g3(m,k,18); c.gst(c.st.cref,3*sidx,prob.x); c.gst(c.st.cref,3*sidx+1,prob.y); c.gst(c.st.cref,3*sidx+2,prob.z); }
        if( ref && !flag ) slide_commit_dense(m, k);
      }
    }
    return nfl;
  }

  /* does this environment have an active contact on a rigid pair?  (multi-word worlds: every pair owns whole words) */
  RKFD_HD bool rigid_active(const ModelDev &m){
    if( Spec::NL != 0 || m.nfw <= 1 ) return RKFD_POPC64(cfl & m.rigid_mask) > 0;
    bool any = false;
    for(int pi=0;pi<m.npair;pi++){
      const PairDev &pr = m.pair[pi]; if( pr.type != C_RIGID ) continue;
      const int nw = (m.cell[pr.cell].nvert + 31) >> 5;
      for(int k=0;k<nw;k++){ flag_select((pr.fofs >> 5) + k); if( cfl & 0x5555555555555555ull ) any = true; }
    }
    return any;
  }
  RKFD_HD void load_flags(){ piv = c.st.piv_type[c.e]; cw = 0; cfl = c.st.cflags[c.e]; }
  RKFD_HD void store_flags(){ c.st.piv_type[c.e] = piv; c.st.cflags[(size_t)(Spec::NL != 0 ? 0 : cw)*c.st.ld + c.e] = cfl; if( bad ) c.st.status[c.e] |= bad;
    if( Ctx::RIGID ){ if( c.st.work ) c.st.work[c.e] = (unsigned char)wk; } }
  /* committed state -> stage state */
  RKFD_HD void load_stage_state(const ModelDev &m){
    const int NQc = Spec::nq(m);
#pragma unroll (Spec::UNROLL)
    for(int j=0;j<NQc;j++){ Tw(rk0+j, c.gld(qc, j)); Tw(rk0+NQc+j, c.gld(qdc, j)); }
  }
  RKFD_HD void evaluate(const ModelDev &m, int stage){
    const bool ref = (stage == ST_REF) || (stage == ST_EVAL_REF);
    /* keep the warps of a block in the same pass: the instruction working set of the SM is then one pass, not
     * the union of all passes (the kernel is far larger than the instruction cache) */
    c.phase_sync(1);
    c.tfence();               /* T-space stores of the previous pass are complete before this pass loads them */
    pass1(m, ref, stage == ST_K1 || stage >= ST_EVAL);
    if constexpr ( Spec::NL == 0 ){ if( m.npair > m.npair_static ) contacts_moving(m, ref); }
    c.phase_sync(2);
    c.tfence();
    if( Ctx::RIGID ){
      /* rigid pairs in contact (reference rkfd_vert.c:385-386): any lane of the warp -> cooperative solve.
       * Round 0 = rkFDUpdateAccBias (rkfd_util.c:149-161): the inward/outward passes without contact forces, then the
       * solve; round 1 = the evaluation proper.  One rolled loop so that the passes exist once in the kernel.
       * Whether round 0 exists is decided per BLOCK and its pieces are separated by block barriers: a warp without
       * contacts skips the work, not the barriers, so that the warps of an SM sit in the same piece of this very large
       * kernel (ncu: 10 instruction-fetch stall cycles per issued instruction when every warp goes its own way).  The
       * Volume solver has barriers inside its solve as well (rkfd_volume.cuh): every warp enters it. */
      wk = 0;
      const unsigned act = c.ballot( rigid_active(m) );
      const bool volume = Spec::NL == 0 && m.solver == S_VOLUME;
      const bool blk = c.block_or(act != 0);
#pragma unroll 1
      for(int round = blk ? 0 : 1; round < 2; round++){
        const bool work = round == 1 || act != 0 || volume;
        if( work ) pass2(m, round ? ref : false);
        c.phase_sync(2);
        c.tfence();
        if( work ) pass3(m, round ? stage : (int)ST_PROBE);
        c.phase_sync(2);
        if( round == 0 ){
          if( work ) rigid_solve(m, ref, act);
          c.gsync();                                   /* lanes leave the solve at different points: reconverge */
          c.phase_sync(2);
        }
      }
      return;
    }
    pass2(m, ref);
    c.phase_sync(2);
    c.tfence();
    pass3(m, stage);
  }
  /* mode 0: rkFDUpdate x nsteps (reference rkfd_sim.c:560-566); mode 1 / 2: a single non-committing /
   * committing evaluation on the committed state (2 = rkFDUpdateInit's t=0 evaluation).  One stage loop so
   * that the evaluation body is instantiated once. */
  RKFD_HD void run(const ModelDev &m, int mode, int nsteps){
    rk0 = Spec::rk_slot(m);
    load_flags();
    const int first = mode == 0 ? ST_K1 : ( mode == 2 ? ST_EVAL_REF : ST_EVAL );
    const int last  = mode == 0 ? ST_REF : first;
    if( mode != 0 ) nsteps = 1;
#pragma unroll 1
    for(int s=0;s<nsteps;s++){
      load_stage_state(m);
      const int ns = m.rk.ns;
      if constexpr ( Spec::FUSE != 0 ){
        /* outward passes [P3(s3) P1(s1)] (Core::outward) and the inward pass of s1 in turn; one loop, one call site each */
#pragma unroll 1
        for(int s3 = -1, s1 = first;;){
          c.phase_sync(1);          /* as in evaluate */
          c.tfence();
          outward(m, s3, s1);
          if( s1 < 0 ) break;
          if( s1 == ST_REF ) commit_swap();   /* pass 3 of the last stage has formed the new state in the output buffer */
          c.phase_sync(2);
          c.tfence();
          pass2(m, s1 == ST_REF || s1 == ST_EVAL_REF);
          s3 = s1; s1 = s1 == last ? -1 : rk_next_stage(s1, ns);
        }
      } else {
#pragma unroll 1
        for(int stage=first;;){
          if( stage == ST_REF ) commit_swap();   /* the output buffer now holds the committed state */
          evaluate(m, stage);
          if( stage == last ) break;
          stage = rk_next_stage(stage, ns);
        }
      }
    }
    store_flags();
  }
};

}  // namespace rkfd
#endif
