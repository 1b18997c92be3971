/* rkfd_b200.h - C-ABI of librokifd_b200.so: the B200-native drop-in for RoKi-FD's rkfd_sim step path.
 *
 * Everything here is plain C (pointers, sizes, PODs).  No CUDA type appears; callers never see the GPU.
 * The entry points are the ones mi-lib/roki-fd v1.7.9 exports for this path, with the same names,
 * argument meaning and error behaviour (NULL / false on failure, rkFDUpdate cannot fail):
 *
 *   this header                         replaces (reference file:line)
 *   ---------------------------------   ---------------------------------------------------------
 *   rkFDCreate / rkFDDestroy            include/roki_fd/rkfd_sim.h:58-59   src/rkfd_sim.c:32,56
 *   rkFDChainReg / RegFile / Unreg      rkfd_sim.h:61-63                   rkfd_sim.c:211,224,237
 *   rkFDChainSetDis / SetVel            rkfd_sim.h:69-70                   rkfd_sim.c:277,283
 *   rkFDContactInfoScanFile             rkfd_sim.h:71                      rkfd_sim.c:259
 *   rkFDUpdateInit / Update / Destroy   rkfd_sim.h:95-97                   rkfd_sim.c:552,560,568
 *   rkFDSolve                           rkfd_sim.h:94                      rkfd_sim.c:576
 *   rkFDODE2Assign / AssignRegular      rkfd_sim.h:85-86 (macros)
 *   rkFDSetSolver(fd, Vert|MLCP|Volume) rkfd_sim.h:89-93 (macro) -> rkFDSolverReset,
 *                                       rkFDSolverCreate_<T>, vtable slot _defci (rkfd_solver.h:23-60)
 *   rkFDPrp + rkFDPrpSet* macros        rkfd_property.h:15-34              rkfd_property.c:10-18
 *   rkFDTime / rkFDDT                   rkfd_sim.h:54-55
 *
 * The reference headers pull ZEDA/ZM/Zeo/RoKi types in by value (zVec, rkChain, rkCD ...).  Those
 * libraries are not part of the reference tree, so this header carries minimal source-compatible
 * stand-ins for exactly the pieces the reference's example programs touch
 * (the .c files of example/chain): zVec, rkChain/rkJoint accessors, rkCDPairChainUnreg.  Programs written
 * against roki_fd.h recompile against this header unchanged (source compatibility; the by-value
 * `rkFD` layout is necessarily different, see INTEGRATION.md).
 *
 * Batched extension (rkFDBatch*): the same create/register/update/destroy life cycle steps B
 * independent copies of the registered world in lockstep on one or more GPUs.
 */
#ifndef ROKI_FD_B200_H
#define ROKI_FD_B200_H

#include <stdbool.h>
#include <stddef.h>
#include <stdio.h>      /* the reference's example programs rely on ZEDA's headers for FILE, BUFSIZ, sprintf, atoi */
#include <stdlib.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __ROKI_FD_EXPORT
#define __ROKI_FD_EXPORT __attribute__((visibility("default")))
#endif

/* ---- defaults (reference include/roki_fd/rkfd_defs.h:15-23) ---------------------------------- */
#define RK_FD_DT_DEFAULT                        0.001
#define RK_FD_CDT_DEFAULT                       0.002
#define RK_FD_JOINT_COMP_K_DEFAULT            100
#define RK_FD_JOINT_COMP_L_DEFAULT              0.01
#define RK_FD_KINETIC_FRICTION_WEIGHT_DEFAULT 100
#define RK_FD_FRICTION_PYRAMID_ORDER_DEFAULT    8
#define RK_FD_MAX_ITER_DEFAULT                 10
#define RK_FD_VEL_EPSILON_DEFAULT              (1.0e-8)

/* ---- ZM / ZEDA stand-ins ---------------------------------------------------------------------- */
typedef struct { int size; double *buf; } zVecStruct;
typedef zVecStruct *zVec;
#define zVecSizeNC(v)    ( (v)->size )
#define zVecSize(v)      ( (v) ? (v)->size : 0 )
#define zVecBufNC(v)     ( (v)->buf )
#define zVecBuf(v)       ( (v)->buf )
#define zVecElemNC(v,i)  ( (v)->buf[i] )
#define zVecElem(v,i)    ( (v)->buf[i] )
#define zVecSetElem(v,i,x) ( (v)->buf[i] = (x) )
#define zDeg2Rad(d)      ( (d) * 3.14159265358979323846 / 180.0 )
#define zRad2Deg(r)      ( (r) * 180.0 / 3.14159265358979323846 )
__ROKI_FD_EXPORT zVec zVecAlloc(int size);
__ROKI_FD_EXPORT void zVecFree(zVec v);
__ROKI_FD_EXPORT void zVecFreeAtOnce(int n, ...);       /* [EXT] ZM: frees n vectors */
__ROKI_FD_EXPORT zVec zVecZero(zVec v);
__ROKI_FD_EXPORT zVec zVecCopy(zVec src, zVec dst);
/* [EXT] ZM zVecFPrint: "<size> ( e0 e1 ... )\n" */
__ROKI_FD_EXPORT void zVecFPrint(FILE *fp, zVec v);
#define zVecPrint(v)     zVecFPrint( stdout, (v) )
/* [EXT] ZEDA zRandInit / zRandF / zRandI: a uniform generator (splitmix64 here; ZEDA's Mersenne-twister stream is not
 * reproduced).  zRandInit seeds from the clock, or from the environment variable ROKIFD_ZRAND_SEED when it is set. */
__ROKI_FD_EXPORT void zRandInit(void);
__ROKI_FD_EXPORT double zRandF(double min, double max);
__ROKI_FD_EXPORT int zRandI(int min, int max);
/* [EXT] ZEDA eprintf: formatted message on stderr */
#define eprintf(...)     fprintf( stderr, __VA_ARGS__ )

typedef struct { double e[3]; } zVec3D;

/* ---- RoKi stand-ins: chain, joint, contact info, collision manager ----------------------------- */
typedef struct _rkChain { void *_b200; } rkChain;
typedef struct _rkJoint rkJoint;          /* opaque handle owned by its chain */
typedef struct { void *_b200; } rkCD;

__ROKI_FD_EXPORT rkChain *rkChainInit(rkChain *chain);
__ROKI_FD_EXPORT void rkChainDestroy(rkChain *chain);
__ROKI_FD_EXPORT rkChain *rkChainClone(rkChain *src, rkChain *dest);
__ROKI_FD_EXPORT rkChain *rkChainReadZTK(rkChain *chain, const char *filename);
__ROKI_FD_EXPORT int rkChainLinkNum(rkChain *chain);
__ROKI_FD_EXPORT int rkChainJointSize(rkChain *chain);
__ROKI_FD_EXPORT rkJoint *rkChainLinkJoint(rkChain *chain, int i);
__ROKI_FD_EXPORT zVec rkChainGetJointDisAll(rkChain *chain, zVec dis);
__ROKI_FD_EXPORT zVec rkChainGetJointVelAll(rkChain *chain, zVec vel);
__ROKI_FD_EXPORT zVec rkChainGetJointAccAll(rkChain *chain, zVec acc);
__ROKI_FD_EXPORT void rkChainSetJointDisAll(rkChain *chain, zVec dis);
__ROKI_FD_EXPORT void rkChainSetJointVelAll(rkChain *chain, zVec vel);
__ROKI_FD_EXPORT int rkJointDOF(rkJoint *joint);
__ROKI_FD_EXPORT void rkJointGetDis(rkJoint *joint, double *val);
__ROKI_FD_EXPORT void rkJointGetVel(rkJoint *joint, double *val);
__ROKI_FD_EXPORT void rkJointGetAcc(rkJoint *joint, double *val);
__ROKI_FD_EXPORT void rkJointMotorSetInput(rkJoint *joint, double *val);
__ROKI_FD_EXPORT void rkCDPairChainUnreg(rkCD *cd, rkChain *chain);
/* collision shapes of a link ([EXT] Zeo zShape3D / RoKi rkCDCell: opaque here).  rkLinkShapeNum / rkLinkShape stand in for RoKi's
 * shape list of a link: shape k of link `link` in the order of the model file (moving links: vertex clouds and box primitives
 * in their file order; static links: their box primitives).  Handles stay valid as long as the chain lives. */
typedef struct _zShape3D zShape3D;
typedef struct _zShape3D rkCDCell;        /* one registered shape = one collision cell */
__ROKI_FD_EXPORT int rkLinkShapeNum(rkChain *chain, int link);
__ROKI_FD_EXPORT zShape3D *rkLinkShape(rkChain *chain, int link, int k);

/* programmatic chain construction (what rkChainReadZTK does from a file) */
enum { RK_B200_JOINT_FIXED = 0, RK_B200_JOINT_REVOL = 1, RK_B200_JOINT_PRISM = 2,
       RK_B200_JOINT_SPHER = 3, RK_B200_JOINT_FLOAT = 4, RK_B200_JOINT_CYLIN = 5, RK_B200_JOINT_HOOKE = 6,
       RK_B200_JOINT_BRFLOAT = 7 };
enum { RK_B200_MOTOR_NONE = 0, RK_B200_MOTOR_DC = 1, RK_B200_MOTOR_TRQ = 2 };
typedef struct {
  const char *name;           /* may be NULL */
  const char *stuff;          /* contact-info key, may be NULL */
  int parent;                 /* link index in this chain, -1 = root; must precede the child */
  int jointtype;
  double frame_R[9];          /* ZTK `frame:` rotation part, row-major */
  double frame_p[3];          /* ZTK `frame:` position part */
  double mass;
  double com[3];
  double inertia[9];          /* about the COM, link axes, row-major */
  double stiffness, viscosity, coulomb, staticfriction;   /* 1-DoF joint passive torque */
  int motortype;
  double motorconstant, admittance, gearratio, rotorinertia, gearinertia, minvoltage, maxvoltage;
  double forcethreshold, torquethreshold;    /* breakable float (example/model/wall.ztk:51-95) */
} rkB200LinkDesc;
__ROKI_FD_EXPORT void rkB200LinkDescInit(rkB200LinkDesc *d);
__ROKI_FD_EXPORT int rkChainB200SetName(rkChain *chain, const char *name);
__ROKI_FD_EXPORT int rkChainB200AddLink(rkChain *chain, const rkB200LinkDesc *d);    /* returns the link index, <0 on error */
__ROKI_FD_EXPORT int rkChainB200LinkAddVerts(rkChain *chain, int link, int nvert, const double *xyz);
__ROKI_FD_EXPORT int rkChainB200LinkAddBox(rkChain *chain, int link, const double center[3], double depth, double width, double height);

/* contact information ([EXT] rkContactInfo; ZTK [roki::contact]) */
enum { RK_CONTACT_RIGID = 0, RK_CONTACT_ELASTIC = 1 };
enum { RK_CONTACT_SF = 0, RK_CONTACT_KF = 1 };
typedef struct {
  char stf[2][32];
  int type;
  double k, l;       /* compensation, relaxation (rigid) */
  double e, v;       /* elasticity, viscosity (elastic)  */
  double sf, kf;     /* static / kinetic friction coefficients */
} rkContactInfo;
typedef struct { int size; rkContactInfo *buf; } rkContactInfoArray;
#define rkContactInfoInit(c)        do{ (c)->stf[0][0] = (c)->stf[1][0] = 0; (c)->type = RK_CONTACT_RIGID; \
                                        (c)->k = (c)->l = (c)->e = (c)->v = (c)->sf = (c)->kf = 0; } while(0)
#define rkContactInfoType(c)        (c)->type
#define rkContactInfoK(c)           (c)->k
#define rkContactInfoL(c)           (c)->l
#define rkContactInfoE(c)           (c)->e
#define rkContactInfoV(c)           (c)->v
#define rkContactInfoSF(c)          (c)->sf
#define rkContactInfoKF(c)          (c)->kf
#define rkContactInfoSetType(c,t)   ( (c)->type = (t) )
#define rkContactInfoSetK(c,x)      ( (c)->k = (x) )
#define rkContactInfoSetL(c,x)      ( (c)->l = (x) )
#define rkContactInfoSetE(c,x)      ( (c)->e = (x) )
#define rkContactInfoSetV(c,x)      ( (c)->v = (x) )
#define rkContactInfoSetSF(c,x)     ( (c)->sf = (x) )
#define rkContactInfoSetKF(c,x)     ( (c)->kf = (x) )

/* ---- properties (reference rkfd_property.h:15-34) --------------------------------------------- */
typedef struct {
  double dt;
  int pyramid;
  double friction_weight;
  int max_iter;
  double vel_eps;
} rkFDPrp;
#define rkFDPrpDT(p)             (p)->dt
#define rkFDPrpPyramid(p)        (p)->pyramid
#define rkFDPrpFrictionWeight(p) (p)->friction_weight
#define rkFDPrpMaxIter(p)        (p)->max_iter
#define rkFDPrpVelEps(p)         (p)->vel_eps
#define rkFDPrpSetDT(f,t)             ( (f)->prp.dt = (t) )
#define rkFDPrpSetPyramid(f,n)        ( (f)->prp.pyramid = (n) )
#define rkFDPrpSetFrictionWeight(f,w) ( (f)->prp.friction_weight = (w) )
#define rkFDPrpSetMaxIter(f,i)        ( (f)->prp.max_iter = (i) )
#define rkFDPrpSetVelEps(f,e)         ( (f)->prp.vel_eps = (e) )
__ROKI_FD_EXPORT bool rkFDPrpInit(rkFDPrp *prp);
__ROKI_FD_EXPORT void rkFDPrpDestroy(rkFDPrp *prp);

/* ---- solver plug-in ABI (reference rkfd_solver.h:23-41) ---------------------------------------- */
struct _rkFDSolver;
typedef struct {
  void (*_defci)(struct _rkFDSolver*, rkContactInfo*);   /* default contact info of the solver          */
  bool (*_init)(struct _rkFDSolver*);                    /* workspace set-up, called by rkFDUpdateInit  */
  void (*_colchk)(struct _rkFDSolver*, bool);            /* collision check of one evaluation           */
  bool (*_update)(struct _rkFDSolver*, bool);            /* joint friction -> penalty -> rigid solve    */
  void (*_update_ref)(struct _rkFDSolver*);              /* previous driving torque bookkeeping         */
  void (*_destroy)(struct _rkFDSolver*);
} rkFDSolverCom;
typedef struct { rkCD cd; } rkFDCD;
#define rkFDCDBase(c) ( (rkCD*)(c) )
typedef struct _rkFDSolver {
  void *prp;
  rkFDSolverCom *com;
  double t;
  rkFDPrp *fdprp;
  rkFDCD *cd;
  void *_b200;     /* owning simulator */
} rkFDSolver;
#define rkFDSolverIsEmpty(s) ( (s)->prp == NULL && (s)->com == NULL )
#define rkFDSolverGetDefaultContactInfo(s,c) (s)->com->_defci(s,c)
#define rkFDSolverUpdateInit(s)              (s)->com->_init(s)
#define rkFDSolverColChk(s,b)                (s)->com->_colchk(s,b)
#define rkFDSolverUpdate(s,b)                (s)->com->_update(s,b)
#define rkFDSolverUpdatePrevDrivingTrq(s)    (s)->com->_update_ref(s)
#define rkFDSolverUpdateDestroy(s)           (s)->com->_destroy(s)
__ROKI_FD_EXPORT void rkFDSolverInit(rkFDSolver *solver);
__ROKI_FD_EXPORT void rkFDSolverReset(rkFDSolver *solver);
__ROKI_FD_EXPORT void rkFDSolverDestroy(rkFDSolver *solver);
__ROKI_FD_EXPORT rkFDSolver *rkFDSolverCreate_Vert(rkFDSolver *s);     /* rkfd_vert.h */
__ROKI_FD_EXPORT rkFDSolver *rkFDSolverCreate_MLCP(rkFDSolver *s);     /* rkfd_mlcp.h */
__ROKI_FD_EXPORT rkFDSolver *rkFDSolverCreate_Volume(rkFDSolver *s);   /* rkfd_volume.h */

/* ---- ODE selection stand-in ([EXT] zODE2Assign / zODE2AssignRegular) ---------------------------- */
enum { RKFD_ODE2_Regular = 0 };
enum { RKFD_ODE_RKG = 0, RKFD_ODE_RK4 = 1, RKFD_ODE_Euler = 2, RKFD_ODE_Heun = 3 };
typedef struct { int form; int integrator; } zODE2;

/* ---- the simulator (reference rkfd_sim.h:24-52) ------------------------------------------------ */
typedef struct { rkChain chain; bool has_rigid_col; bool done_abi_init; } rkFDChain;
typedef struct {
  rkFDChain fc;
  int _offset;
  zVecStruct _dis, _vel, _acc;
} rkFDCellDat;
typedef struct _rkFDCell { struct _rkFDCell *prev, *next; rkFDCellDat data; } rkFDCell;
typedef struct { int size; rkFDCell root; } rkFDCellList;
#define rkFDCellDatChain(d) ( (rkChain*)&(d)->fc )
#define rkFDCellChain(c)    rkFDCellDatChain(&(c)->data)

typedef struct _rkFD {
  double t;
  rkFDPrp prp;
  rkFDSolver solver;
  rkFDCellList list;
  rkContactInfoArray ci;
  rkContactInfo cidef;
  rkFDCD cd;
  zODE2 ode;
  int ode_step;
  zVec dis, vel;
  zVec acc;
  int size;
  void *_b200;      /* device engine + host bookkeeping (opaque) */
} rkFD;

#define rkFDTime(f)   (f)->t
#define rkFDDT(f)     (f)->prp.dt
#define rkFDGetPrp(f) ( &(f)->prp )

__ROKI_FD_EXPORT rkFD *rkFDCreate(rkFD *fd);
__ROKI_FD_EXPORT void rkFDDestroy(rkFD *fd);
__ROKI_FD_EXPORT rkFDCell *rkFDChainReg(rkFD *fd, rkChain *chain);
__ROKI_FD_EXPORT rkFDCell *rkFDChainRegFile(rkFD *fd, char filename[]);
__ROKI_FD_EXPORT bool rkFDChainUnreg(rkFD *fd, rkFDCell *cell);
__ROKI_FD_EXPORT void rkFDChainSetDis(rkFDCell *lc, zVec dis);
__ROKI_FD_EXPORT void rkFDChainSetVel(rkFDCell *lc, zVec vel);
__ROKI_FD_EXPORT bool rkFDContactInfoScanFile(rkFD *fd, char filename[]);
/* for a fake-crawler (reference rkfd_sim.h:73-80, rkfd_sim.c:386-440): a cell in slide mode behaves like a belt running with
 * `vel` about `axis` (frame of the cell's link): its surface velocity enters the relative contact velocity
 * (rkFDLinkAddSlideVel, rkfd_util.c:26-40) and the anchors of sticking contacts ride on it (rkFDUpdateRefSlide, :218-237).
 * The shape must belong to the chain of a registered cell (rkFDCellChain), and the calls must precede rkFDUpdateInit. */
__ROKI_FD_EXPORT void rkFDCDCellSetSlideMode(rkCDCell *cell, bool mode);
__ROKI_FD_EXPORT void rkFDCDCellSetSlideVel(rkCDCell *cell, double vel);
__ROKI_FD_EXPORT void rkFDCDCellSetSlideAxis(rkCDCell *cell, zVec3D *axis);
__ROKI_FD_EXPORT rkCDCell *rkFDShape3DGetCDCell(rkFD *fd, zShape3D *shape);
__ROKI_FD_EXPORT rkCDCell *rkFDShape3DSetSlideMode(rkFD *fd, zShape3D *shape, bool mode);
__ROKI_FD_EXPORT rkCDCell *rkFDShape3DSetSlideVel(rkFD *fd, zShape3D *shape, double vel);
__ROKI_FD_EXPORT rkCDCell *rkFDShape3DSetSlideAxis(rkFD *fd, zShape3D *shape, zVec3D *axis);
__ROKI_FD_EXPORT zVec rkFDODECatDefault(zVec x, double k, zVec v, zVec xnew, void *util);
__ROKI_FD_EXPORT zVec rkFDODESubDefault(zVec x1, zVec x2, zVec dx, void *util);
#define rkFDODE2Assign(f,t)        ( (f)->ode.form = RKFD_ODE2_##t )
#define rkFDODE2AssignRegular(f,t) ( (f)->ode.integrator = RKFD_ODE_##t )
#define rkFDSetSolver(f,type) do{                                 \
    rkFDSolverReset( &(f)->solver );                              \
    rkFDSolverCreate_##type( &(f)->solver );                      \
    rkFDSolverGetDefaultContactInfo( &(f)->solver, &(f)->cidef ); \
  } while(0)
__ROKI_FD_EXPORT rkFD *rkFDSolve(rkFD *fd);
__ROKI_FD_EXPORT void rkFDUpdateInit(rkFD *fd);
__ROKI_FD_EXPORT rkFD *rkFDUpdate(rkFD *fd);
__ROKI_FD_EXPORT void rkFDUpdateDestroy(rkFD *fd);

/* programmatic counterpart of rkFDContactInfoScanFile: appends one [roki::contact] record */
__ROKI_FD_EXPORT bool rkFDContactInfoAdd(rkFD *fd, const char *stuff_a, const char *stuff_b, int type,
                                         double k, double l, double e, double v, double sf, double kf);

/* ---- batched extension -------------------------------------------------------------------------
 * Host arrays are environment-major: q[B][size], u[B][links], contact arrays [B][slots](x3).
 * All return 0 on success, non-zero on error (message through rkFDBatchLastError). */
__ROKI_FD_EXPORT int rkFDBatchSetEnvNum(rkFD *fd, int B);                       /* before rkFDUpdateInit; default 1 */
__ROKI_FD_EXPORT int rkFDBatchSetDevices(rkFD *fd, const int *ids, int n);      /* before rkFDUpdateInit; default current */
__ROKI_FD_EXPORT int rkFDBatchSetStream(rkFD *fd, void *cuda_stream);           /* after rkFDUpdateInit; single device */
__ROKI_FD_EXPORT int rkFDBatchReady(rkFD *fd);                                  /* 1 when the device engine exists */
__ROKI_FD_EXPORT int rkFDBatchEnvNum(rkFD *fd);
__ROKI_FD_EXPORT int rkFDBatchLinkNum(rkFD *fd);                                /* moving links per env */
__ROKI_FD_EXPORT int rkFDBatchContactSlotNum(rkFD *fd);
__ROKI_FD_EXPORT int rkFDBatchSetState(rkFD *fd, const double *q, const double *qd);
__ROKI_FD_EXPORT int rkFDBatchGetState(rkFD *fd, double *q, double *qd, double *qdd);
__ROKI_FD_EXPORT int rkFDBatchSetMotorInput(rkFD *fd, const double *u);
__ROKI_FD_EXPORT int rkFDBatchGetContactForce(rkFD *fd, double *f);
/* Volume solver (reference rkfd_volume.c: one 6-D wrench per rigid pair instead of vertex forces): the first three slots of a
 * pair hold the pair wrench of the last committing evaluation - force, torque about the volume centre (world axes) - and the
 * volume centre */
__ROKI_FD_EXPORT int rkFDBatchGetContactState(rkFD *fd, int *active, int *type, double *ref);
__ROKI_FD_EXPORT int rkFDBatchSetContactState(rkFD *fd, const int *active, const int *type, const double *ref);
__ROKI_FD_EXPORT int rkFDBatchGetPivot(rkFD *fd, int *type, double *prev_trq);
__ROKI_FD_EXPORT int rkFDBatchSetPivot(rkFD *fd, const int *type, const double *prev_trq);
__ROKI_FD_EXPORT int rkFDBatchGetStatus(rkFD *fd, int *status);                 /* per env, bit0: non-finite acceleration */
/* Environment re-sort.  The kernels address environments by slot (thread index) and environments never interact, so the
 * engine re-orders the slots by the number of active contact vertices - under the Vert / Volume solvers by the work class of
 * the environment's last rigid solve - every `steps` steps (default in worlds with contact pairs: 16; rigid pairs under the
 * Vert solver 4, under the Volume solver 1; RKFD_RESORT=<steps> overrides): warps then hold environments with the same
 * amount of contact work.
 * Results per environment do not depend on it and every host-side call maps through the order; only callers of
 * rkFDBatchDevicePtr see slots: they read the order with rkFDBatchSlotMap (perm[slot] = environment of that shard, B
 * entries) or switch the re-sort off (steps = 0: slot = environment). */
__ROKI_FD_EXPORT int rkFDBatchSetResortInterval(rkFD *fd, int steps);
__ROKI_FD_EXPORT int rkFDBatchSlotMap(rkFD *fd, int shard, int *perm);
__ROKI_FD_EXPORT long long rkFDBatchResortCount(rkFD *fd);
__ROKI_FD_EXPORT long long rkFDBatchResortKernelCount(rkFD *fd);     /* kernels the re-sorts launched so far (beside rkFDBatchLaunchCount's step kernels) */
/* end-of-run statistics of the batch, reduced on the device; sums: out[0] environments, [1] environments with an active
 * contact, [2] active contact vertices, [3] environments with a non-zero status word; maxima: [4] |q''|, [5] |q'|;
 * [6..7] reserved (0).  A one-process-per-GPU job all-reduces [0..3] with SUM and [4..5] with MAX (SURVEY.md section 8e:
 * the only collective of the path, after the run). */
__ROKI_FD_EXPORT int rkFDBatchStats(rkFD *fd, double out[8]);
__ROKI_FD_EXPORT int rkFDBatchEval(rkFD *fd, int do_up_ref);                    /* one evaluation on the committed state */
__ROKI_FD_EXPORT rkFD *rkFDUpdateN(rkFD *fd, int k);                            /* k steps in one launch, asynchronous */
__ROKI_FD_EXPORT int rkFDBatchSync(rkFD *fd);
/* asynchronous transfers for pipelined callers: host buffers must be pinned and stay valid until rkFDBatchSync;
 * copies run on dedicated streams and overlap the step kernels of neighbouring steps.  rkFDBatchJoin makes the
 * compute stream wait for all queued copies. */
__ROKI_FD_EXPORT int rkFDBatchSetStateAsync(rkFD *fd, const double *q, const double *qd);
__ROKI_FD_EXPORT int rkFDBatchSetMotorInputAsync(rkFD *fd, const double *u);
__ROKI_FD_EXPORT int rkFDBatchGetStateAsync(rkFD *fd, double *q, double *qd, double *qdd);
__ROKI_FD_EXPORT int rkFDBatchJoin(rkFD *fd);
__ROKI_FD_EXPORT void *rkFDBatchDevicePtr(rkFD *fd, int shard, int which, int *ld, int *B);  /* 0 q, 1 qd, 2 qdd, 3 u; SoA [k][ld] */
__ROKI_FD_EXPORT long long rkFDBatchLaunchCount(rkFD *fd);
/* Environment reset: restarts some environments of a running batch while the others go on.  After the call, environment
 * envs[i] is bit for bit what environment i of a new simulator of the same world would be after an rkFDUpdateInit from
 * (q[i], qd[i], u[i]): state, q'' of the committing evaluation at t=0, contact flags, anchors and forces, friction pivots,
 * broken breakable-float joints (broken again only if the t=0 evaluation breaks them) and status word - right after the call
 * and in every later step.  Environments not listed are unaffected.  fd->t does not change (nothing on the step path reads
 * the time).  Both calls need rkFDUpdateInit; n = 0 does nothing.  Each call runs one step-kernel launch per shard touched and
 * up to 65,536 environments (counted in rkFDBatchLaunchCount), with a few small kernels around it
 * (rkFDBatchResetKernelCount).
 * rkFDBatchResetEnvs: host arrays, env-major: q[n][size] (required), qd[n][size] (NULL: zero), u[n][links] (NULL: keep the
 * current input); global environment indices.  Everything is checked before any device work (indices in [0, B), no
 * duplicates, q given): a refused call changes nothing.  Synchronous, like rkFDBatchSetState.
 * rkFDBatchResetEnvsDevice: the same arrays on the device of shard `shard` (envs[n], q[n][size], ...), indices local to
 * that shard (slots do not matter: the engine maps them through its re-sort order).  Stream-ordered on the engine's stream
 * without a host synchronisation, except for the first call and a call with a longer list than any before (it allocates the
 * reset's buffers).  Indices outside [0, B) are skipped; a duplicate index is the caller's error (the environment ends up with
 * one of its states). */
__ROKI_FD_EXPORT int rkFDBatchResetEnvs(rkFD *fd, int n, const int *envs, const double *q, const double *qd, const double *u);
__ROKI_FD_EXPORT int rkFDBatchResetEnvsDevice(rkFD *fd, int shard, int n, const int *envs, const double *q, const double *qd, const double *u);
__ROKI_FD_EXPORT long long rkFDBatchResetKernelCount(rkFD *fd);       /* gather, zero fill and scatter launches of the resets so far */
/* Link kinematics: world frames and velocities of selected links of every environment, from the committed state (what
 * rkFDBatchGetState returns: q and q' of the current buffer, and for breakable-float joints the broken bit of rkFDBatchGetPivot).
 * The frames are computed from the committed q with the joint model of the step kernel's pass 1 (revolute sin/cos from
 * sincos(q)): they agree with the step kernel's internal frames to rounding.  Nothing of the engine's state is written.
 * links: host array of nlink link indices in [0, rkFDBatchLinkNum) - moving chains in registration order, links in chain order
 * (the order of the motor input u); duplicates are allowed; NULL: all links, then nlink must be rkFDBatchLinkNum.  nlink = 0
 * does nothing.  nlink < 0, nlink > 32 (MAX_LINKS) or an index out of range is refused, and nothing is written.
 * frame[env][k][12]: the world-from-link rotation R of links[k], row-major, then the world position p of the link origin.
 * vel[env][k][6]: the linear velocity of the link origin, then the angular velocity, both in world axes.
 * Either pointer may be NULL: that output is neither computed nor written.  An unbroken breakable-float joint contributes no
 * joint velocity (it is rigid).
 * rkFDBatchGetLinkFrames: host arrays, global environment index, every shard; synchronous, like rkFDBatchGetState.
 * rkFDBatchGetLinkFramesDevice: device buffers on the device of shard `shard`, [Bs][nlink][12] and [Bs][nlink][6], indexed by
 * the environment local to the shard (the engine maps its re-sorted slots itself).  Stream-ordered on the engine's stream,
 * without a host synchronisation or an allocation.
 * Both need rkFDUpdateInit; each launches one kernel per shard it covers (rkFDBatchLinkFrameKernelCount). */
__ROKI_FD_EXPORT int rkFDBatchGetLinkFrames(rkFD *fd, int nlink, const int *links, double *frame, double *vel);
__ROKI_FD_EXPORT int rkFDBatchGetLinkFramesDevice(rkFD *fd, int shard, int nlink, const int *links, double *frame, double *vel);
__ROKI_FD_EXPORT long long rkFDBatchLinkFrameKernelCount(rkFD *fd);   /* kinematics launches of the calls so far */
/* External wrenches: a force and a torque applied to links of every environment, for pushes, disturbances, tethers, drag or
 * forces from another model.  The reference has no such input (it clears every link's wrench list at each evaluation).
 * rkFDBatchSetExtWrenchLinks declares which links take one, before rkFDUpdateInit: links[0..n) are link indices in
 * [0, rkFDBatchLinkNum), in the order of the motor input, without duplicates, 0 <= n <= 32; n = 0 clears the declaration.  A
 * refused call (after rkFDUpdateInit, an index out of range, a duplicate, n out of range) changes nothing.  A new declaration
 * drops a wrench held as pending.  Without a declaration nothing of the model, of the kernel choice or of the step changes.
 * A declared world runs the generic kernels: the serial-arm specialisations take no external wrench.
 * rkFDBatchSetExtWrench: host memory, env-major w[B][n][6] = (force, torque) of declared link k in row k.  The force acts at the
 * link's centre of mass and the torque is about the centre of mass, both in world axes.  A push f at another world point p
 * adds (p - c) x f to the torque, c being the world position of the centre of mass.  Before rkFDUpdateInit the wrench is held
 * as pending, so the committing evaluation at t = 0 sees it; afterwards it is synchronous, like rkFDBatchSetMotorInput.
 * rkFDBatchSetExtWrenchDevice: a device buffer [Bs][n][6] on the device of shard `shard`, indexed by the environment local to the
 * shard (the engine maps it to its re-sorted slot); stream-ordered on the engine's stream, without a host synchronisation or an
 * allocation.  It needs rkFDUpdateInit.
 * Like the motor input, the wrench is an input held until it is changed; it is zero until set.  It is constant over the
 * evaluations of a step (the stage evaluations and the committing one) and enters rkFDBatchEval as well.  It enters every
 * contact solver (penalty, MLCP, Vert, Volume), through the bias of the articulated-body pass, and the transmitted-wrench test of
 * breakable-float joints.  rkFDBatchResetEnvs* keeps it: a reset environment restarts as a new simulator given its current
 * wrench before rkFDUpdateInit.  A non-finite wrench ends up in the status word (bit 0) like any other non-finite acceleration.
 * Both setters need a declaration. */
__ROKI_FD_EXPORT int rkFDBatchSetExtWrenchLinks(rkFD *fd, int n, const int *links);
__ROKI_FD_EXPORT int rkFDBatchSetExtWrench(rkFD *fd, const double *w);
__ROKI_FD_EXPORT int rkFDBatchSetExtWrenchDevice(rkFD *fd, int shard, const double *w);
/* The compiled step-kernel variant that shard `shard` launches, as chosen by rkFDUpdateInit from the model and the tuning
 * variables RKFD_SPEC, RKFD_FORCE_BLOCK, RKFD_FORCE_MINB, RKFD_FORCE_GSCR and RKFD_FORCE_SMEM: v[0] threads per block, v[1] 1
 * when the scratch column lives in device memory (0: shared memory), v[2] 1 for the rigid-contact kernels, v[3] the model
 * specialisation id (0: the generic table-driven kernel), v[4] the minimum resident blocks per SM it was compiled for.
 * Needs rkFDUpdateInit; a bad shard index is refused. */
__ROKI_FD_EXPORT int rkFDBatchKernelVariant(rkFD *fd, int shard, int v[5]);
/* the flattened model of the last rkFDUpdateInit as text (host side; also after an rkFDUpdateInit that found no device):
 * returns the length needed */
__ROKI_FD_EXPORT int rkFDB200DescribeModel(rkFD *fd, char *buf, int cap);
__ROKI_FD_EXPORT const char *rkFDBatchLastError(void);
__ROKI_FD_EXPORT int rkFDBatchDeviceCount(void);
/* measured fp64 FMA roofline of the current device in TFLOP/s (register-resident DFMA loop on all SMs) */
__ROKI_FD_EXPORT int rkFDB200MeasureFp64(double *tflops);

/* ---- function forms of the reference's struct-poking macros, for FFI callers (ctypes, cgo ...) that
 * cannot expand C macros: rkFD storage, rkFDPrpSet*, rkFDSetSolver, rkFDTime, rkFDCellChain ------------ */
__ROKI_FD_EXPORT rkFD *rkFDB200Alloc(void);                                  /* calloc(sizeof(rkFD)); free with rkFDB200Free */
__ROKI_FD_EXPORT void rkFDB200Free(rkFD *fd);
__ROKI_FD_EXPORT rkChain *rkChainB200Alloc(void);
__ROKI_FD_EXPORT void rkChainB200Free(rkChain *chain);
__ROKI_FD_EXPORT void rkFDB200PrpSet(rkFD *fd, double dt, int pyramid, double friction_weight, int max_iter);
__ROKI_FD_EXPORT int rkFDB200SetSolver(rkFD *fd, int solver);                /* 0 Vert, 1 MLCP, 2 Volume */
__ROKI_FD_EXPORT int rkFDB200SetIntegrator(rkFD *fd, int integrator);        /* RKFD_ODE_RKG / RK4 / Euler / Heun: rkFDODE2AssignRegular */
__ROKI_FD_EXPORT double rkFDB200Time(rkFD *fd);
__ROKI_FD_EXPORT int rkFDB200Size(rkFD *fd);
__ROKI_FD_EXPORT rkChain *rkFDB200CellChain(rkFDCell *cell);
__ROKI_FD_EXPORT const double *rkFDB200Dis(rkFD *fd);
__ROKI_FD_EXPORT const double *rkFDB200Vel(rkFD *fd);
__ROKI_FD_EXPORT const double *rkFDB200Acc(rkFD *fd);

#ifdef __cplusplus
}
#endif
#endif /* ROKI_FD_B200_H */
