/* rkfd_capi.cpp - the C-ABI of librokifd_b200.so (include/roki_fd/rkfd_b200.h).
 *
 * Host-side mirror of the reference's simulator object: registration bookkeeping, state vectors,
 * solver plug-in table, life cycle (reference src/rkfd_sim.c:32-70, 79-255, 277-287, 552-582,
 * src/rkfd_solver.c:10-34, src/rkfd_property.c:10-18).  All arithmetic of the step path runs on the
 * GPU through rkfd::Engine; nothing here computes dynamics and there is no CPU fallback.
 */
#include "roki_fd/rkfd_b200.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstdarg>
#include <cstring>
#include <ctime>
#include <stdexcept>
#include <string>
#include <vector>

#include "rkfd_engine.h"
#include "rkfd_math.cuh"
#include "rkfd_model.h"
#include "rkfd_ztk.h"

using namespace rkfd;

struct _rkJoint { struct ChainImpl *chain; int link; };

struct FDImpl;
struct _zShape3D { struct ChainImpl *chain; int link, cell; };     /* a shape of a link = one collision cell */
struct ChainImpl : ChainHost {
  std::vector<_rkJoint> joints;
  std::vector<_zShape3D*> shapes;       /* handles given out by rkLinkShape (owned; a clone starts without any) */
  ChainImpl() = default;
  ChainImpl(const ChainImpl &o) : ChainHost(o), joints(o.joints), owner(o.owner), link_base(o.link_base), q_base(o.q_base) {}
  ChainImpl &operator=(const ChainImpl &) = delete;
  ~ChainImpl(){ for(_zShape3D *s : shapes) delete s; }
  FDImpl *owner = nullptr;     /* set for the clone held by a registered cell */
  int link_base = 0;           /* first global (moving) link index of this chain in the engine, -1 if static */
  int q_base = 0;
  void refresh(){ sync_sizes(); joints.resize(links.size()); for(size_t i=0;i<links.size();i++){ joints[i].chain = this; joints[i].link = (int)i; } }
};

struct FDImpl {
  std::vector<rkFDCell*> cells;          /* registration order */
  std::vector<ContactInfoHost> ci;
  int B = 1; bool batch = false; std::vector<int> devices; int resort = -1;     /* -1: the engine's default */
  Engine *engine = nullptr;
  ModelDev model;
  std::vector<double> pend_q, pend_qd, pend_u;   /* batched initial state given before rkFDUpdateInit */
  std::vector<int> fext_links;                   /* links declared for an external wrench (rkFDBatchSetExtWrenchLinks) */
  std::vector<double> pend_w;                    /* external wrench given before rkFDUpdateInit */
  std::vector<int> mp_links;                     /* links declared for per-environment mass properties (rkFDBatchSetMassPropLinks) */
  std::vector<double> pend_mp;                   /* mass properties given before rkFDUpdateInit */
  bool warned = false;
};

static thread_local std::string g_err;
static int fail(const std::string &m){ g_err = m; return 1; }
static void complain(const char *where, const std::string &m){ g_err = m; std::fprintf(stderr, "rokifd_b200: %s: %s\n", where, m.c_str()); }

static ChainImpl *CI(rkChain *c){ return c ? (ChainImpl*)c->_b200 : nullptr; }
static FDImpl *FI(rkFD *fd){ return fd ? (FDImpl*)fd->_b200 : nullptr; }

/* ---- zVec ------------------------------------------------------------------------------------ */
extern "C" zVec zVecAlloc(int size)
{
  zVec v = (zVec)std::calloc(1, sizeof(zVecStruct)); if( !v ) return NULL;
  v->size = size; v->buf = (double*)std::calloc(size > 0 ? size : 1, sizeof(double));
  if( !v->buf ){ std::free(v); return NULL; }
  return v;
}
extern "C" void zVecFree(zVec v){ if( v ){ std::free(v->buf); std::free(v); } }
extern "C" void zVecFreeAtOnce(int n, ...){ va_list ap; va_start(ap, n); for(int i=0;i<n;i++) zVecFree(va_arg(ap, zVec)); va_end(ap); }
extern "C" zVec zVecZero(zVec v){ if( v ) std::memset(v->buf, 0, v->size*sizeof(double)); return v; }
extern "C" zVec zVecCopy(zVec s, zVec d){ if( !s || !d || s->size != d->size ) return NULL; std::memcpy(d->buf, s->buf, s->size*sizeof(double)); return d; }

extern "C" void zVecFPrint(FILE *fp, zVec v)
{
  if( !fp ) return;
  if( !v ){ std::fprintf(fp, "(null vector)\n"); return; }
  std::fprintf(fp, "%d (", v->size);
  for(int i=0;i<v->size;i++) std::fprintf(fp, " %.10g", v->buf[i]);
  std::fprintf(fp, " )\n");
}
/* [EXT] ZEDA random numbers: splitmix64 */
static unsigned long long g_rand_state = 0x9E3779B97F4A7C15ull;
static unsigned long long rand_next(){ unsigned long long z = (g_rand_state += 0x9E3779B97F4A7C15ull); z = (z ^ (z >> 30))*0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27))*0x94D049BB133111EBull; return z ^ (z >> 31); }
extern "C" void zRandInit(void){ const char *s = std::getenv("ROKIFD_ZRAND_SEED"); g_rand_state = s ? std::strtoull(s, NULL, 10) : (unsigned long long)std::time(NULL); }
extern "C" double zRandF(double min, double max){ return min + (max - min)*((double)(rand_next() >> 11)*(1.0/9007199254740992.0)); }
extern "C" int zRandI(int min, int max){ return max <= min ? min : min + (int)(rand_next() % (unsigned long long)(max - min + 1)); }

/* ---- chain stand-in ---------------------------------------------------------------------------- */
extern "C" rkChain *rkChainInit(rkChain *c){ if( !c ) return NULL; ChainImpl *ci = new ChainImpl; ci->refresh(); c->_b200 = ci; return c; }
extern "C" void rkChainDestroy(rkChain *c){ if( c && c->_b200 ){ delete CI(c); c->_b200 = NULL; } }
extern "C" rkChain *rkChainClone(rkChain *src, rkChain *dst)
{
  if( !CI(src) || !dst ) return NULL;
  ChainImpl *n = new ChainImpl(*CI(src)); n->owner = nullptr; n->refresh(); dst->_b200 = n; return dst;
}
extern "C" rkChain *rkChainReadZTK(rkChain *c, const char *filename)
{
  if( !c ) return NULL;
  ChainImpl *ci = new ChainImpl; std::string err;
  if( !ztk_read_chain(filename, *ci, err) ){ complain("rkChainReadZTK", err); delete ci; c->_b200 = NULL; return NULL; }
  ci->refresh(); c->_b200 = ci; return c;
}
extern "C" int rkChainLinkNum(rkChain *c){ return CI(c) ? (int)CI(c)->links.size() : 0; }
extern "C" int rkChainJointSize(rkChain *c){ return CI(c) ? CI(c)->joint_size() : 0; }
extern "C" rkJoint *rkChainLinkJoint(rkChain *c, int i){ ChainImpl *ci = CI(c); if( !ci || i < 0 || i >= (int)ci->links.size() ) return NULL; return &ci->joints[i]; }
static zVec get_all(rkChain *c, zVec v, int which)
{
  ChainImpl *ci = CI(c); if( !ci || !v ) return NULL;
  const std::vector<double> &s = which == 0 ? ci->dis : ( which == 1 ? ci->vel : ci->acc );
  for(int i=0;i<v->size && i<(int)s.size();i++) v->buf[i] = s[i];
  return v;
}
extern "C" zVec rkChainGetJointDisAll(rkChain *c, zVec v){ return get_all(c, v, 0); }
extern "C" zVec rkChainGetJointVelAll(rkChain *c, zVec v){ return get_all(c, v, 1); }
extern "C" zVec rkChainGetJointAccAll(rkChain *c, zVec v){ return get_all(c, v, 2); }
extern "C" void rkChainSetJointDisAll(rkChain *c, zVec v){ ChainImpl *ci = CI(c); if( !ci || !v ) return; for(int i=0;i<v->size && i<(int)ci->dis.size();i++) ci->dis[i] = v->buf[i]; }
extern "C" void rkChainSetJointVelAll(rkChain *c, zVec v){ ChainImpl *ci = CI(c); if( !ci || !v ) return; for(int i=0;i<v->size && i<(int)ci->vel.size();i++) ci->vel[i] = v->buf[i]; }
extern "C" int rkJointDOF(rkJoint *j){ return j ? jtype_ndof(j->chain->links[j->link].jtype) : 0; }
static void joint_get(rkJoint *j, double *val, int which)
{
  if( !j || !val ) return;
  ChainImpl *ci = j->chain; const int o = ci->link_qofs(j->link), n = jtype_ndof(ci->links[j->link].jtype);
  const std::vector<double> &s = which == 0 ? ci->dis : ( which == 1 ? ci->vel : ci->acc );
  for(int k=0;k<n;k++) val[k] = s[o+k];
}
extern "C" void rkJointGetDis(rkJoint *j, double *v){ joint_get(j, v, 0); }
extern "C" void rkJointGetVel(rkJoint *j, double *v){ joint_get(j, v, 1); }
extern "C" void rkJointGetAcc(rkJoint *j, double *v){ joint_get(j, v, 2); }
extern "C" void rkJointMotorSetInput(rkJoint *j, double *val)
{
  if( !j || !val ) return;
  ChainImpl *ci = j->chain; ci->motor_in[j->link] = *val;
  FDImpl *fi = ci->owner;
  if( fi && fi->engine && ci->link_base >= 0 ){
    try { fi->engine->fill_rows(2, ci->link_base + j->link, 1, val); }      /* the row u[link][0..B) in one fill */
    catch(const std::exception &ex){ complain("rkJointMotorSetInput", ex.what()); }
  }
}
/* [EXT] RoKi rk_cd: drops the collision pairs between the cells of `chain` itself (registered by default, as in the reference:
 * example/chain/boxdrop_test.c:37, arm_box_test.c:49).  Pairs are formed in rkFDUpdateInit: call it before. */
extern "C" void rkCDPairChainUnreg(rkCD *cd, rkChain *chain){ (void)cd; if( CI(chain) ) CI(chain)->self_collide = false; }

/* ---- shapes / collision cells and their slide mode (reference rkfd_sim.c:386-440) ---------------- */
static int link_cell_num(const ChainImpl *ci, int link){ const LinkHost &l = ci->links[link]; return ci->is_static() ? (int)l.boxes.size() : (int)l.shapes.size(); }
extern "C" int rkLinkShapeNum(rkChain *chain, int link){ ChainImpl *ci = CI(chain); return ( ci && link >= 0 && link < (int)ci->links.size() ) ? link_cell_num(ci, link) : 0; }
extern "C" zShape3D *rkLinkShape(rkChain *chain, int link, int k)
{
  ChainImpl *ci = CI(chain); if( !ci || link < 0 || link >= (int)ci->links.size() || k < 0 || k >= link_cell_num(ci, link) ) return NULL;
  for(_zShape3D *s : ci->shapes) if( s->link == link && s->cell == k ) return s;
  _zShape3D *s = new _zShape3D{ci, link, k}; ci->shapes.push_back(s); return s;
}
static LinkHost::Slide *cell_slide(rkCDCell *cell, const char *where)
{
  if( !cell || !cell->chain ) return nullptr;
  ChainImpl *ci = cell->chain;
  if( ci->owner && ci->owner->engine ){ complain(where, "slide mode must be set before rkFDUpdateInit"); return nullptr; }
  LinkHost &l = ci->links[cell->link];
  for(LinkHost::Slide &s : l.slides) if( s.cell == cell->cell ) return &s;
  LinkHost::Slide s; s.cell = cell->cell; s.mode = false; s.vel = 0.0; s.axis[0] = s.axis[1] = s.axis[2] = 0.0;
  l.slides.push_back(s); return &l.slides.back();
}
extern "C" void rkFDCDCellSetSlideMode(rkCDCell *cell, bool mode){ if( LinkHost::Slide *s = cell_slide(cell, "rkFDCDCellSetSlideMode") ) s->mode = mode; }
extern "C" void rkFDCDCellSetSlideVel(rkCDCell *cell, double vel){ if( LinkHost::Slide *s = cell_slide(cell, "rkFDCDCellSetSlideVel") ) s->vel = vel; }
extern "C" void rkFDCDCellSetSlideAxis(rkCDCell *cell, zVec3D *axis){ if( !axis ) return; if( LinkHost::Slide *s = cell_slide(cell, "rkFDCDCellSetSlideAxis") ){ s->axis[0] = axis->e[0]; s->axis[1] = axis->e[1]; s->axis[2] = axis->e[2]; } }

extern "C" rkCDCell *rkFDShape3DGetCDCell(rkFD *fd, zShape3D *shape)
{
  FDImpl *fi = FI(fd); if( !fi || !shape ) return NULL;
  for(rkFDCell *c : fi->cells) if( CI(&c->data.fc.chain) == shape->chain ) return shape;       /* the cell of a registered chain's shape */
  return NULL;
}
extern "C" rkCDCell *rkFDShape3DSetSlideMode(rkFD *fd, zShape3D *shape, bool mode){ rkCDCell *c = rkFDShape3DGetCDCell(fd, shape); if( c ) rkFDCDCellSetSlideMode(c, mode); return c; }
extern "C" rkCDCell *rkFDShape3DSetSlideVel(rkFD *fd, zShape3D *shape, double vel){ rkCDCell *c = rkFDShape3DGetCDCell(fd, shape); if( c ) rkFDCDCellSetSlideVel(c, vel); return c; }
extern "C" rkCDCell *rkFDShape3DSetSlideAxis(rkFD *fd, zShape3D *shape, zVec3D *axis){ rkCDCell *c = rkFDShape3DGetCDCell(fd, shape); if( c ) rkFDCDCellSetSlideAxis(c, axis); return c; }

extern "C" void rkB200LinkDescInit(rkB200LinkDesc *d)
{
  std::memset(d, 0, sizeof *d); d->parent = -1; d->frame_R[0] = d->frame_R[4] = d->frame_R[8] = 1.0;
  d->gearratio = 1.0; d->minvoltage = -1e300; d->maxvoltage = 1e300;
}
extern "C" int rkChainB200SetName(rkChain *c, const char *name){ if( !CI(c) ) return 1; CI(c)->name = name ? name : ""; return 0; }
extern "C" int rkChainB200AddLink(rkChain *c, const rkB200LinkDesc *d)
{
  ChainImpl *ci = CI(c); if( !ci || !d ) return -1;
  if( d->parent >= (int)ci->links.size() ){ g_err = "parent must precede child"; return -1; }
  LinkHost l; l.name = d->name ? d->name : ""; l.stuff = d->stuff ? d->stuff : ""; l.parent = d->parent; l.jtype = d->jointtype;
  std::memcpy(l.Ro, d->frame_R, sizeof l.Ro); std::memcpy(l.po, d->frame_p, sizeof l.po);
  l.mass = d->mass; std::memcpy(l.com, d->com, sizeof l.com); std::memcpy(l.inertia, d->inertia, sizeof l.inertia);
  l.stiffness = d->stiffness; l.viscosity = d->viscosity; l.coulomb = d->coulomb; l.sfriction = d->staticfriction;
  l.brk_f = d->forcethreshold; l.brk_t = d->torquethreshold;
  l.motor.type = d->motortype; l.motor.k = d->motorconstant; l.motor.admittance = d->admittance; l.motor.gear = d->gearratio;
  l.motor.rotor_inertia = d->rotorinertia; l.motor.gear_inertia = d->gearinertia; l.motor.min = d->minvoltage; l.motor.max = d->maxvoltage;
  ci->links.push_back(l); ci->refresh();
  return (int)ci->links.size() - 1;
}
extern "C" int rkChainB200LinkAddVerts(rkChain *c, int link, int nvert, const double *xyz)
{
  ChainImpl *ci = CI(c); if( !ci || link < 0 || link >= (int)ci->links.size() || nvert <= 0 || !xyz ) return 1;
  ci->links[link].shapes.push_back(std::vector<double>(xyz, xyz + 3*nvert)); return 0;
}
extern "C" int rkChainB200LinkAddBox(rkChain *c, int link, const double center[3], double depth, double width, double height)
{
  ChainImpl *ci = CI(c); if( !ci || link < 0 || link >= (int)ci->links.size() ) return 1;
  BoxShape b; std::memcpy(b.center, center, sizeof b.center); b.depth = depth; b.width = width; b.height = height;
  b.cloud = (int)ci->links[link].shapes.size();
  ci->links[link].boxes.push_back(b);
  /* a box on a moving link collides through its 8 corners ([EXT] zeo box -> polyhedron) */
  std::vector<double> v;
  for(int k=0;k<8;k++){ v.push_back(center[0] + ((k&1)?0.5:-0.5)*depth); v.push_back(center[1] + ((k&2)?0.5:-0.5)*width); v.push_back(center[2] + ((k&4)?0.5:-0.5)*height); }
  ci->links[link].shapes.push_back(v);
  return 0;
}

/* ---- properties / solver table ------------------------------------------------------------------ */
extern "C" bool rkFDPrpInit(rkFDPrp *prp)
{
  prp->dt = RK_FD_DT_DEFAULT; prp->pyramid = RK_FD_FRICTION_PYRAMID_ORDER_DEFAULT;
  prp->friction_weight = RK_FD_KINETIC_FRICTION_WEIGHT_DEFAULT; prp->max_iter = RK_FD_MAX_ITER_DEFAULT;
  prp->vel_eps = RK_FD_VEL_EPSILON_DEFAULT; return true;
}
extern "C" void rkFDPrpDestroy(rkFDPrp *prp){ (void)prp; }

extern "C" void rkFDSolverInit(rkFDSolver *s){ s->prp = NULL; s->com = NULL; s->t = 0; s->fdprp = NULL; s->cd = NULL; s->_b200 = NULL; }
extern "C" void rkFDSolverReset(rkFDSolver *s){ if( s->prp ) std::free(s->prp); s->prp = NULL; s->com = NULL; }
extern "C" void rkFDSolverDestroy(rkFDSolver *s){ rkFDSolverReset(s); rkFDSolverInit(s); }

/* default contact info of the three solvers (reference rkfd_vert.c:340-348, rkfd_mlcp.c:301-310, rkfd_volume.c:961-969) */
static void solver_defci(rkFDSolver *s, rkContactInfo *ci)
{
  (void)s; rkContactInfoInit(ci); rkContactInfoSetType(ci, RK_CONTACT_RIGID);
  rkContactInfoSetK(ci, 1000.0); rkContactInfoSetL(ci, 1.0); rkContactInfoSetSF(ci, 0.5); rkContactInfoSetKF(ci, 0.3);
}
/* The device solvers are fused into the step kernel; the per-stage slots drive whole evaluations. */
static bool solver_init(rkFDSolver *s){ (void)s; return true; }
static void solver_colchk(rkFDSolver *s, bool b){ (void)s; (void)b; }
static bool solver_update(rkFDSolver *s, bool do_up_ref)
{
  rkFD *fd = (rkFD*)s->_b200; FDImpl *fi = FI(fd); if( !fi || !fi->engine ) return false;
  try { fi->engine->eval(do_up_ref); fi->engine->sync(); } catch(const std::exception &ex){ complain("rkFDSolverUpdate", ex.what()); return false; }
  return true;
}
static void solver_update_ref(rkFDSolver *s){ (void)s; }
static void solver_destroy(rkFDSolver *s){ (void)s; }
static rkFDSolverCom g_solver_vert   = { solver_defci, solver_init, solver_colchk, solver_update, solver_update_ref, solver_destroy };
static rkFDSolverCom g_solver_mlcp   = { solver_defci, solver_init, solver_colchk, solver_update, solver_update_ref, solver_destroy };
static void solver_defci_volume(rkFDSolver *s, rkContactInfo *ci){ solver_defci(s, ci); rkContactInfoSetL(ci, 0.001); }   /* rkfd_volume.c:961-969 */
static rkFDSolverCom g_solver_volume = { solver_defci_volume, solver_init, solver_colchk, solver_update, solver_update_ref, solver_destroy };
static rkFDSolver *solver_create(rkFDSolver *s, rkFDSolverCom *com){ if( !(s->prp = std::calloc(1, 64)) ) return NULL; s->com = com; return s; }
extern "C" rkFDSolver *rkFDSolverCreate_Vert(rkFDSolver *s){ return solver_create(s, &g_solver_vert); }
extern "C" rkFDSolver *rkFDSolverCreate_MLCP(rkFDSolver *s){ return solver_create(s, &g_solver_mlcp); }
extern "C" rkFDSolver *rkFDSolverCreate_Volume(rkFDSolver *s){ return solver_create(s, &g_solver_volume); }

/* ---- simulator life cycle ------------------------------------------------------------------------- */
extern "C" rkFD *rkFDCreate(rkFD *fd)
{
  if( !fd ) return NULL;
  fd->t = 0.0; rkFDPrpInit(&fd->prp);
  fd->list.size = 0; fd->list.root.prev = fd->list.root.next = &fd->list.root;
  fd->ci.size = 0; fd->ci.buf = NULL; fd->cd.cd._b200 = NULL;
  fd->size = 0; fd->dis = fd->vel = fd->acc = NULL;
  rkFDODE2Assign(fd, Regular); rkFDODE2AssignRegular(fd, RKG); fd->ode_step = 0;
  fd->_b200 = new FDImpl;
  rkFDSolverInit(&fd->solver); fd->solver.t = 0; fd->solver.fdprp = &fd->prp; fd->solver.cd = &fd->cd; fd->solver._b200 = fd;
  rkFDSetSolver(fd, Vert);
  return fd;
}

static void destroy_engine(FDImpl *fi){ delete fi->engine; fi->engine = nullptr; }

extern "C" void rkFDDestroy(rkFD *fd)
{
  FDImpl *fi = FI(fd); if( !fi ) return;
  destroy_engine(fi);
  rkFDSolverDestroy(&fd->solver);
  zVecFree(fd->dis); zVecFree(fd->vel); zVecFree(fd->acc); fd->dis = fd->vel = fd->acc = NULL;
  std::free(fd->ci.buf); fd->ci.buf = NULL; fd->ci.size = 0;
  for(rkFDCell *c : fi->cells){ rkChainDestroy(rkFDCellChain(c)); std::free(c); }
  delete fi; fd->_b200 = NULL; fd->size = 0; fd->list.size = 0;
}

/* rebuilds fd->dis/vel/acc and every cell's window after a registration change
 * (reference _rkFDAllocJointStatePush/Pop, rkfd_sim.c:79-155) */
static bool relayout(rkFD *fd)
{
  FDImpl *fi = FI(fd); int size = 0, lbase = 0;
  for(rkFDCell *c : fi->cells) size += CI(rkFDCellChain(c))->joint_size();
  zVec nd = zVecAlloc(size), nv = zVecAlloc(size), na = zVecAlloc(size);
  if( !nd || !nv || !na ){ zVecFree(nd); zVecFree(nv); zVecFree(na); return false; }
  int off = 0;
  fd->list.root.next = fd->list.root.prev = &fd->list.root;
  for(rkFDCell *c : fi->cells){
    ChainImpl *ci = CI(rkFDCellChain(c)); const int n = ci->joint_size();
    for(int k=0;k<n;k++){ nd->buf[off+k] = ci->dis[k]; nv->buf[off+k] = ci->vel[k]; }
    c->data._offset = off; c->data._dis.size = c->data._vel.size = c->data._acc.size = n;
    c->data._dis.buf = nd->buf + off; c->data._vel.buf = nv->buf + off; c->data._acc.buf = na->buf + off;
    ci->q_base = off; ci->link_base = ci->is_static() ? -1 : lbase; if( !ci->is_static() ) lbase += (int)ci->links.size();
    off += n;
    c->prev = fd->list.root.prev; c->next = &fd->list.root; fd->list.root.prev->next = c; fd->list.root.prev = c;
  }
  zVecFree(fd->dis); zVecFree(fd->vel); zVecFree(fd->acc);
  fd->dis = nd; fd->vel = nv; fd->acc = na; fd->size = size; fd->list.size = (int)fi->cells.size();
  return true;
}

static rkFDCell *cell_push(rkFD *fd, ChainImpl *ci)
{
  FDImpl *fi = FI(fd);
  rkFDCell *c = (rkFDCell*)std::calloc(1, sizeof(rkFDCell));
  if( !c ){ delete ci; return NULL; }
  ci->owner = fi; ci->refresh();
  c->data.fc.chain._b200 = ci; c->data.fc.has_rigid_col = false; c->data.fc.done_abi_init = false;
  fi->cells.push_back(c);
  if( !relayout(fd) ){ complain("rkFDChainReg", "cannot allocate joint state"); rkFDDestroy(fd); return NULL; }
  return c;
}
extern "C" rkFDCell *rkFDChainReg(rkFD *fd, rkChain *chain)
{
  if( !FI(fd) || !CI(chain) ) return NULL;
  if( FI(fd)->engine ){ complain("rkFDChainReg", "registration after rkFDUpdateInit is not supported"); return NULL; }
  return cell_push(fd, new ChainImpl(*CI(chain)));          /* the chain is cloned (reference rkfd_sim.c:217) */
}
extern "C" rkFDCell *rkFDChainRegFile(rkFD *fd, char filename[])
{
  if( !FI(fd) ) return NULL;
  if( FI(fd)->engine ){ complain("rkFDChainRegFile", "registration after rkFDUpdateInit is not supported"); return NULL; }
  ChainImpl *ci = new ChainImpl; std::string err;
  if( !ztk_read_chain(filename, *ci, err) ){ complain("rkFDChainRegFile", err); delete ci; return NULL; }
  return cell_push(fd, ci);
}
extern "C" bool rkFDChainUnreg(rkFD *fd, rkFDCell *cell)
{
  FDImpl *fi = FI(fd); if( !fi ) return false;
  /* the engine holds the flattened model: the reference sizes its solver and pair arrays in rkFDUpdateInit as well
   * (rkfd_sim.c:479-490) - unregister between rkFDUpdateDestroy and the next rkFDUpdateInit */
  if( fi->engine ){ complain("rkFDChainUnreg", "unregistration after rkFDUpdateInit is not supported (call rkFDUpdateDestroy first)"); return false; }
  for(size_t i=0;i<fi->cells.size();i++) if( fi->cells[i] == cell ){
    fi->cells.erase(fi->cells.begin()+i);
    rkChainDestroy(rkFDCellChain(cell)); std::free(cell);
    if( !relayout(fd) ){ rkFDDestroy(fd); return false; }
    return true;
  }
  return false;
}
/* On a running simulator the cell windows of the reference alias fd->dis/vel (rkfd_sim.c:277-287): a SetDis/SetVel between
 * two updates changes the state the next step integrates from.  Here that state lives on the device: the cell's slice is
 * written to it for every environment (reset / teleport callers). */
static void push_cell_state(rkFDCell *lc, int which)
{
  ChainImpl *ci = CI(rkFDCellChain(lc)); FDImpl *fi = ci ? ci->owner : nullptr;
  if( !fi || !fi->engine || ci->is_static() ) return;
  const int n = lc->data._dis.size; if( n <= 0 ) return;
  try { fi->engine->fill_rows(which, ci->q_base, n, which == 0 ? lc->data._dis.buf : lc->data._vel.buf); }
  catch(const std::exception &ex){ complain(which == 0 ? "rkFDChainSetDis" : "rkFDChainSetVel", ex.what()); }
}
extern "C" void rkFDChainSetDis(rkFDCell *lc, zVec dis)
{
  if( !lc || !dis ) return;
  ChainImpl *ci = CI(rkFDCellChain(lc));
  for(int k=0;k<dis->size && k<lc->data._dis.size;k++){ lc->data._dis.buf[k] = dis->buf[k]; ci->dis[k] = dis->buf[k]; }
  push_cell_state(lc, 0);
}
extern "C" void rkFDChainSetVel(rkFDCell *lc, zVec vel)
{
  if( !lc || !vel ) return;
  ChainImpl *ci = CI(rkFDCellChain(lc));
  for(int k=0;k<vel->size && k<lc->data._vel.size;k++){ lc->data._vel.buf[k] = vel->buf[k]; ci->vel[k] = vel->buf[k]; }
  push_cell_state(lc, 1);
}

static void ci_to_public(rkFD *fd)
{
  FDImpl *fi = FI(fd);
  std::free(fd->ci.buf); fd->ci.size = (int)fi->ci.size();
  fd->ci.buf = (rkContactInfo*)std::calloc(fi->ci.size() ? fi->ci.size() : 1, sizeof(rkContactInfo));
  for(size_t i=0;i<fi->ci.size();i++){
    rkContactInfo &c = fd->ci.buf[i]; const ContactInfoHost &h = fi->ci[i];
    std::snprintf(c.stf[0], sizeof c.stf[0], "%s", h.a.c_str()); std::snprintf(c.stf[1], sizeof c.stf[1], "%s", h.b.c_str());
    c.type = h.type; c.k = h.K; c.l = h.L; c.e = h.E; c.v = h.V; c.sf = h.SF; c.kf = h.KF;
  }
}
extern "C" bool rkFDContactInfoScanFile(rkFD *fd, char filename[])
{
  FDImpl *fi = FI(fd); if( !fi ) return false;
  std::vector<ContactInfoHost> ci; std::string err;
  if( !ztk_read_contact_info(filename, ci, err) ){ complain("rkFDContactInfoScanFile", err); return false; }
  fi->ci = ci; ci_to_public(fd);       /* an earlier table is replaced (reference rkfd_sim.c:262-264) */
  return true;
}
extern "C" bool rkFDContactInfoAdd(rkFD *fd, const char *a, const char *b, int type, double k, double l, double e, double v, double sf, double kf)
{
  FDImpl *fi = FI(fd); if( !fi || !a || !b ) return false;
  ContactInfoHost c; c.a = a; c.b = b; c.type = type; c.K = k; c.L = l; c.E = e; c.V = v; c.SF = sf; c.KF = kf;
  fi->ci.push_back(c); ci_to_public(fd); return true;
}

/* host mirror of the committed state of environment 0 (what a scalar caller reads after rkFDUpdate) */
static void mirror_env0(rkFD *fd)
{
  FDImpl *fi = FI(fd); if( !fi->engine || fd->size == 0 ) return;
  const int n = fd->size; std::vector<double> q((size_t)fi->B*n), qd((size_t)fi->B*n), qdd((size_t)fi->B*n);
  fi->engine->get_state(q.data(), qd.data(), qdd.data());
  for(int k=0;k<n;k++){ fd->dis->buf[k] = q[k]; fd->vel->buf[k] = qd[k]; fd->acc->buf[k] = qdd[k]; }
  for(rkFDCell *c : fi->cells){
    ChainImpl *ci = CI(rkFDCellChain(c)); const int o = c->data._offset;
    for(int k=0;k<(int)ci->dis.size();k++){ ci->dis[k] = q[o+k]; ci->vel[k] = qd[o+k]; ci->acc[k] = qdd[o+k]; }
  }
}

extern "C" void rkFDUpdateInit(rkFD *fd)
{
  FDImpl *fi = FI(fd); if( !fi ) return;
  try {
    destroy_engine(fi);
    WorldHost w;
    for(rkFDCell *c : fi->cells) w.chains.push_back(CI(rkFDCellChain(c)));
    w.ci = fi->ci;
    w.cidef.type = fd->cidef.type; w.cidef.K = fd->cidef.k; w.cidef.L = fd->cidef.l; w.cidef.E = fd->cidef.e; w.cidef.V = fd->cidef.v;
    w.cidef.SF = fd->cidef.sf; w.cidef.KF = fd->cidef.kf;
    w.dt = fd->prp.dt; w.friction_weight = fd->prp.friction_weight; w.pyramid = fd->prp.pyramid; w.max_iter = fd->prp.max_iter;
    w.solver = fd->solver.com == &g_solver_mlcp ? S_MLCP : ( fd->solver.com == &g_solver_volume ? S_VOLUME : S_VERT );
    if( fd->ode.form != RKFD_ODE2_Regular || fd->ode.integrator < RKFD_ODE_RKG || fd->ode.integrator > RKFD_ODE_Heun )
      throw std::runtime_error("integrators: Regular form with RKG, RK4, Euler or Heun");
    w.integrator = fd->ode.integrator;
    w.fext_links = fi->fext_links;
    w.mp_links = fi->mp_links;
    std::string err; std::vector<double> mp_default;
    if( !build_model(w, fi->model, err, &mp_default) ) throw std::runtime_error(err);
    /* static chains carry no joint state, so the device rows are the host offsets of relayout() */
    if( fi->model.nq != fd->size ) throw std::runtime_error("joint state layout mismatch between the host mirror and the device model");
    fi->engine = new Engine(fi->model, fi->B, fi->devices, mp_default.data());
    if( fi->resort >= 0 ) fi->engine->set_resort_interval(fi->resort);
    const int n = fd->size, nl = fi->model.nl, B = fi->B;
    /* initial state: the batched arrays when given, else the scalar state replicated over the envs */
    std::vector<double> q((size_t)B*n), qd((size_t)B*n), u((size_t)B*(nl > 0 ? nl : 1), 0.0);
    if( (int)fi->pend_q.size() == B*n && n > 0 ){ q = fi->pend_q; qd = fi->pend_qd; }
    else for(int e=0;e<B;e++) for(int k=0;k<n;k++){ q[(size_t)e*n+k] = fd->dis->buf[k]; qd[(size_t)e*n+k] = fd->vel->buf[k]; }
    if( (int)fi->pend_u.size() == B*nl && nl > 0 ) u = fi->pend_u;
    else for(rkFDCell *c : fi->cells){ ChainImpl *ci = CI(rkFDCellChain(c)); if( ci->link_base < 0 ) continue;
      for(int e=0;e<B;e++) for(size_t k=0;k<ci->links.size();k++) u[(size_t)e*nl + ci->link_base + k] = ci->motor_in[k]; }
    if( n > 0 ) fi->engine->set_state(q.data(), qd.data());
    if( nl > 0 ) fi->engine->set_motor_input(u.data());
    if( fi->model.nfext > 0 && fi->pend_w.size() == (size_t)B*6*fi->model.nfext ) fi->engine->set_ext_wrench(fi->pend_w.data());
    if( fi->model.nmp > 0 && fi->pend_mp.size() == (size_t)B*10*fi->model.nmp ) fi->engine->set_mass_prop(fi->pend_mp.data());
    fi->engine->eval(true);            /* the committing evaluation at t=0 (reference rkfd_sim.c:556) */
    if( !fi->batch ){ fi->engine->sync(); mirror_env0(fd); }
  } catch(const std::exception &ex){ complain("rkFDUpdateInit", ex.what()); destroy_engine(fi); }
}

extern "C" rkFD *rkFDUpdateN(rkFD *fd, int k)
{
  FDImpl *fi = FI(fd); if( !fi ) return fd;
  /* NULL and a message on EVERY call: `while( rkFDTime(&fd) < T ) rkFDUpdate(&fd);` would otherwise spin on a time that never
   * advances; the time is pushed to +inf as well so that such loops end even when the return value is ignored */
  if( !fi->engine ){ complain("rkFDUpdate", "no device engine (rkFDUpdateInit failed or was not called; there is no CPU fallback)"); fd->t = HUGE_VAL; return NULL; }
  try {
    fi->engine->step(k);
    fd->t += k*fd->prp.dt; fd->solver.t = fd->t;
    if( !fi->batch ){ fi->engine->sync(); mirror_env0(fd); }
  } catch(const std::exception &ex){ complain("rkFDUpdate", ex.what()); }
  return fd;
}
extern "C" rkFD *rkFDUpdate(rkFD *fd){ return rkFDUpdateN(fd, 1); }
extern "C" void rkFDUpdateDestroy(rkFD *fd){ FDImpl *fi = FI(fd); if( !fi ) return; try { if( fi->engine ) fi->engine->sync(); } catch(...){} destroy_engine(fi); }
extern "C" rkFD *rkFDSolve(rkFD *fd){ rkFDUpdateInit(fd); rkFDUpdate(fd); rkFDUpdateDestroy(fd); return fd; }

/* joint-space increment on the configuration manifold (reference rkfd_sim.c:306-336 + [EXT] rkChainCatJointDisAll) */
extern "C" zVec rkFDODECatDefault(zVec x, double k, zVec v, zVec xnew, void *util)
{
  rkFD *fd = (rkFD*)util; FDImpl *fi = FI(fd); if( !fi || !x || !v || !xnew ) return NULL;
  for(int i=0;i<x->size;i++) xnew->buf[i] = x->buf[i];
  for(rkFDCell *c : fi->cells){
    ChainImpl *ci = CI(rkFDCellChain(c)); int o = c->data._offset;
    for(const LinkHost &l : ci->links){
      const int n = jtype_ndof(l.jtype); double *xi = xnew->buf + o; const double *vi = v->buf + o;
      if( l.jtype == J_SPHER || l.jtype == J_FLOAT ){
        const int r = l.jtype == J_FLOAT ? 3 : 0;
        for(int a=0;a<r;a++) xi[a] += k*vi[a];
        const V3 aa = aa_cascade(v3(xi[r],xi[r+1],xi[r+2]), v3(k*vi[r],k*vi[r+1],k*vi[r+2]));
        xi[r] = aa.x; xi[r+1] = aa.y; xi[r+2] = aa.z;
      } else for(int a=0;a<n;a++) xi[a] += k*vi[a];
      o += n;
    }
  }
  return xnew;
}
extern "C" zVec rkFDODESubDefault(zVec x1, zVec x2, zVec dx, void *util)
{
  rkFD *fd = (rkFD*)util; FDImpl *fi = FI(fd); if( !fi || !x1 || !x2 || !dx ) return NULL;
  for(int i=0;i<x1->size;i++) dx->buf[i] = x1->buf[i];
  for(rkFDCell *c : fi->cells){
    ChainImpl *ci = CI(rkFDCellChain(c)); int o = c->data._offset;
    for(const LinkHost &l : ci->links){
      const int n = jtype_ndof(l.jtype); double *di = dx->buf + o; const double *yi = x2->buf + o;
      if( l.jtype == J_SPHER || l.jtype == J_FLOAT ){
        const int r = l.jtype == J_FLOAT ? 3 : 0;
        for(int a=0;a<r;a++) di[a] -= yi[a];
        /* d = log( R(x1) R(x2)^T ): the increment w with x1 = cat(x2, 1, w) */
        const V3 d = aa_cascade(v3(-yi[r],-yi[r+1],-yi[r+2]), v3(di[r],di[r+1],di[r+2]));
        di[r] = d.x; di[r+1] = d.y; di[r+2] = d.z;
      } else for(int a=0;a<n;a++) di[a] -= yi[a];
      o += n;
    }
  }
  return dx;
}

/* ---- batched extension ---------------------------------------------------------------------------- */
#define BATCH_GUARD(fd) FDImpl *fi = FI(fd); if( !fi ) return fail("not a created rkFD")
#define NEED_ENGINE() if( !fi->engine ) return fail("rkFDUpdateInit has not been called (or failed)")
#define TRY(stmt) try { stmt; } catch(const std::exception &ex){ return fail(ex.what()); } return 0

extern "C" int rkFDBatchSetEnvNum(rkFD *fd, int B){ BATCH_GUARD(fd); if( fi->engine ) return fail("set the environment count before rkFDUpdateInit"); if( B <= 0 ) return fail("B must be positive"); fi->B = B; fi->batch = true; return 0; }
extern "C" int rkFDBatchSetDevices(rkFD *fd, const int *ids, int n){ BATCH_GUARD(fd); if( fi->engine ) return fail("set the devices before rkFDUpdateInit"); fi->devices.assign(ids, ids + (n > 0 ? n : 0)); return 0; }
extern "C" int rkFDBatchSetStream(rkFD *fd, void *stream){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->set_stream(stream)); }
extern "C" int rkFDBatchReady(rkFD *fd){ FDImpl *fi = FI(fd); return ( fi && fi->engine ) ? 1 : 0; }
extern "C" int rkFDBatchEnvNum(rkFD *fd){ FDImpl *fi = FI(fd); return fi ? fi->B : 0; }
extern "C" int rkFDBatchLinkNum(rkFD *fd){ FDImpl *fi = FI(fd); if( !fi ) return 0; int n = 0; for(rkFDCell *c : fi->cells){ ChainImpl *ci = CI(rkFDCellChain(c)); if( !ci->is_static() ) n += (int)ci->links.size(); } return n; }
extern "C" int rkFDBatchContactSlotNum(rkFD *fd){ FDImpl *fi = FI(fd); return ( fi && fi->engine ) ? fi->model.nslot : 0; }
extern "C" int rkFDBatchSetState(rkFD *fd, const double *q, const double *qd)
{
  BATCH_GUARD(fd);
  if( !fi->engine ){ const size_t n = (size_t)fi->B*fd->size; if( !q || !qd ) return fail("q and qd are both needed before rkFDUpdateInit");
    fi->pend_q.assign(q, q+n); fi->pend_qd.assign(qd, qd+n); return 0; }
  TRY(fi->engine->set_state(q, qd));
}
extern "C" int rkFDBatchGetState(rkFD *fd, double *q, double *qd, double *qdd){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->get_state(q, qd, qdd)); }
extern "C" int rkFDBatchSetMotorInput(rkFD *fd, const double *u)
{
  BATCH_GUARD(fd);
  if( !fi->engine ){ const size_t n = (size_t)fi->B*rkFDBatchLinkNum(fd); fi->pend_u.assign(u, u+n); return 0; }
  TRY(fi->engine->set_motor_input(u));
}
extern "C" int rkFDBatchGetContactForce(rkFD *fd, double *f){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->get_contact(NULL, NULL, NULL, f)); }
extern "C" int rkFDBatchGetContactState(rkFD *fd, int *a, int *t, double *r){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->get_contact(a, t, r, NULL)); }
extern "C" int rkFDBatchSetContactState(rkFD *fd, const int *a, const int *t, const double *r){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->set_contact(a, t, r)); }
extern "C" int rkFDBatchGetPivot(rkFD *fd, int *t, double *p){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->get_pivot(t, p)); }
extern "C" int rkFDBatchSetPivot(rkFD *fd, const int *t, const double *p){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->set_pivot(t, p)); }
extern "C" int rkFDBatchGetStatus(rkFD *fd, int *s){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->get_status(s)); }
/* environment re-sort (rkfd_engine.cu): slots ordered by contact count every `steps` steps; 0 = never (slot = environment) */
extern "C" int rkFDBatchSetResortInterval(rkFD *fd, int steps){ BATCH_GUARD(fd); if( steps < 0 ) return fail("steps must be >= 0"); fi->resort = steps; if( fi->engine ) fi->engine->set_resort_interval(steps); return 0; }
extern "C" int rkFDBatchSlotMap(rkFD *fd, int shard, int *perm){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->slot_map(shard, perm)); }
extern "C" long long rkFDBatchResortCount(rkFD *fd){ FDImpl *fi = FI(fd); return ( fi && fi->engine ) ? fi->engine->resorts() : 0; }
extern "C" long long rkFDBatchResortKernelCount(rkFD *fd){ FDImpl *fi = FI(fd); return ( fi && fi->engine ) ? fi->engine->resort_kernels() : 0; }
/* end-of-run statistics of the whole batch, reduced on the device (SURVEY.md section 8e: what a multi-process job all-reduces) */
extern "C" int rkFDBatchStats(rkFD *fd, double out[8]){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->stats(out)); }
extern "C" int rkFDBatchEval(rkFD *fd, int ref){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->eval(ref != 0)); }
extern "C" int rkFDBatchSetStateAsync(rkFD *fd, const double *q, const double *qd){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->set_state_async(q, qd)); }
extern "C" int rkFDBatchSetMotorInputAsync(rkFD *fd, const double *u){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->set_motor_input_async(u)); }
extern "C" int rkFDBatchGetStateAsync(rkFD *fd, double *q, double *qd, double *qdd){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->get_state_async(q, qd, qdd)); }
extern "C" int rkFDBatchJoin(rkFD *fd){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->join()); }
extern "C" int rkFDBatchSync(rkFD *fd){ BATCH_GUARD(fd); NEED_ENGINE(); TRY(fi->engine->sync()); }
extern "C" void *rkFDBatchDevicePtr(rkFD *fd, int shard, int which, int *ld, int *B){ FDImpl *fi = FI(fd); if( !fi || !fi->engine ) return NULL; return fi->engine->device_ptr(shard, which, ld, B); }
extern "C" long long rkFDBatchLaunchCount(rkFD *fd){ FDImpl *fi = FI(fd); return ( fi && fi->engine ) ? fi->engine->launches() : 0; }
/* environment reset (Engine::reset_envs): the listed environments restart as in a new rkFDUpdateInit, the others go on */
extern "C" int rkFDBatchResetEnvs(rkFD *fd, int n, const int *envs, const double *q, const double *qd, const double *u)
{
  BATCH_GUARD(fd); NEED_ENGINE();
  if( n < 0 ) return fail("rkFDBatchResetEnvs: n must be >= 0");
  if( n == 0 ) return 0;
  if( !envs || !q ) return fail("rkFDBatchResetEnvs: envs and q are needed");
  std::vector<char> seen(fi->B, 0);
  for(int i=0;i<n;i++){
    const int e = envs[i];
    if( e < 0 || e >= fi->B ) return fail("rkFDBatchResetEnvs: environment " + std::to_string(e) + " out of range [0, " + std::to_string(fi->B) + ")");
    if( seen[e] ) return fail("rkFDBatchResetEnvs: environment " + std::to_string(e) + " listed twice");
    seen[e] = 1;
  }
  try {
    fi->engine->reset_envs_host(n, envs, q, qd, u);
    if( !fi->batch ) mirror_env0(fd);
  } catch(const std::exception &ex){ return fail(ex.what()); }
  return 0;
}
extern "C" int rkFDBatchResetEnvsDevice(rkFD *fd, int shard, int n, const int *envs, const double *q, const double *qd, const double *u)
{
  BATCH_GUARD(fd); NEED_ENGINE();
  if( shard < 0 || shard >= fi->engine->num_shards() ) return fail("rkFDBatchResetEnvsDevice: shard index out of range");
  if( n < 0 ) return fail("rkFDBatchResetEnvsDevice: n must be >= 0");
  if( n > 0 && ( !envs || !q ) ) return fail("rkFDBatchResetEnvsDevice: envs and q are needed");
  TRY(fi->engine->reset_envs(shard, n, envs, q, qd, u));
}
extern "C" long long rkFDBatchResetKernelCount(rkFD *fd){ FDImpl *fi = FI(fd); return ( fi && fi->engine ) ? fi->engine->reset_kernels() : 0; }
/* link kinematics (Engine::link_frames): world frames and velocities of selected links from the committed state */
extern "C" int rkFDBatchGetLinkFrames(rkFD *fd, int nlink, const int *links, double *frame, double *vel)
{
  BATCH_GUARD(fd); NEED_ENGINE();
  KinDev t; std::string err;
  if( !kin_table(fi->engine->model(), nlink, links, t, err) ) return fail("rkFDBatchGetLinkFrames: " + err);
  TRY(fi->engine->link_frames_host(t, frame, vel));
}
extern "C" int rkFDBatchGetLinkFramesDevice(rkFD *fd, int shard, int nlink, const int *links, double *frame, double *vel)
{
  BATCH_GUARD(fd); NEED_ENGINE();
  if( shard < 0 || shard >= fi->engine->num_shards() ) return fail("rkFDBatchGetLinkFramesDevice: shard index out of range");
  KinDev t; std::string err;
  if( !kin_table(fi->engine->model(), nlink, links, t, err) ) return fail("rkFDBatchGetLinkFramesDevice: " + err);
  TRY(fi->engine->link_frames(shard, t, frame, vel));
}
extern "C" long long rkFDBatchLinkFrameKernelCount(rkFD *fd){ FDImpl *fi = FI(fd); return ( fi && fi->engine ) ? fi->engine->link_frame_kernels() : 0; }
/* net contact wrench on selected links (Engine::link_contact_wrench): what the last committing evaluation pushed onto them */
extern "C" int rkFDBatchGetLinkContactWrench(rkFD *fd, int nlink, const int *links, double *w)
{
  BATCH_GUARD(fd); NEED_ENGINE();
  LcwDev t; std::string err;
  if( !link_contact_table(fi->engine->model(), nlink, links, t, err) ) return fail("rkFDBatchGetLinkContactWrench: " + err);
  if( nlink > 0 && !w ) return fail("rkFDBatchGetLinkContactWrench: w is needed");
  TRY(fi->engine->link_contact_wrench_host(t, w));
}
extern "C" int rkFDBatchGetLinkContactWrenchDevice(rkFD *fd, int shard, int nlink, const int *links, double *w)
{
  BATCH_GUARD(fd); NEED_ENGINE();
  if( shard < 0 || shard >= fi->engine->num_shards() ) return fail("rkFDBatchGetLinkContactWrenchDevice: shard index out of range");
  LcwDev t; std::string err;
  if( !link_contact_table(fi->engine->model(), nlink, links, t, err) ) return fail("rkFDBatchGetLinkContactWrenchDevice: " + err);
  if( nlink > 0 && !w ) return fail("rkFDBatchGetLinkContactWrenchDevice: w is needed");
  TRY(fi->engine->link_contact_wrench(shard, t, w));
}
extern "C" long long rkFDBatchLinkContactKernelCount(rkFD *fd){ FDImpl *fi = FI(fd); return ( fi && fi->engine ) ? fi->engine->link_contact_kernels() : 0; }
/* external wrenches on declared links (Engine::set_ext_wrench): an input held like the motor input */
extern "C" int rkFDBatchSetExtWrenchLinks(rkFD *fd, int n, const int *links)
{
  BATCH_GUARD(fd);
  if( fi->engine ) return fail("rkFDBatchSetExtWrenchLinks: declare the links before rkFDUpdateInit");
  if( n < 0 || n > MAX_LINKS ) return fail("rkFDBatchSetExtWrenchLinks: n must be in [0, " + std::to_string(MAX_LINKS) + "]");
  if( n > 0 && !links ) return fail("rkFDBatchSetExtWrenchLinks: links is needed");
  const int nl = rkFDBatchLinkNum(fd);
  std::vector<char> seen(nl > 0 ? nl : 1, 0);
  for(int k=0;k<n;k++){
    const int i = links[k];
    if( i < 0 || i >= nl ) return fail("rkFDBatchSetExtWrenchLinks: link " + std::to_string(i) + " out of range [0, " + std::to_string(nl) + ")");
    if( seen[i] ) return fail("rkFDBatchSetExtWrenchLinks: link " + std::to_string(i) + " listed twice");
    seen[i] = 1;
  }
  fi->fext_links.assign(links, links + n);
  fi->pend_w.clear();                 /* a wrench held for an earlier declaration has another row count */
  return 0;
}
extern "C" int rkFDBatchSetExtWrench(rkFD *fd, const double *w)
{
  BATCH_GUARD(fd);
  if( fi->fext_links.empty() ) return fail("rkFDBatchSetExtWrench: no link is declared (rkFDBatchSetExtWrenchLinks)");
  if( !w ) return fail("rkFDBatchSetExtWrench: w is needed");
  if( !fi->engine ){ fi->pend_w.assign(w, w + (size_t)fi->B*6*fi->fext_links.size()); return 0; }
  TRY(fi->engine->set_ext_wrench(w));
}
extern "C" int rkFDBatchSetExtWrenchDevice(rkFD *fd, int shard, const double *w)
{
  BATCH_GUARD(fd); NEED_ENGINE();
  if( fi->engine->model().nfext <= 0 ) return fail("rkFDBatchSetExtWrenchDevice: no link is declared (rkFDBatchSetExtWrenchLinks)");
  if( shard < 0 || shard >= fi->engine->num_shards() ) return fail("rkFDBatchSetExtWrenchDevice: shard index out of range");
  if( !w ) return fail("rkFDBatchSetExtWrenchDevice: w is needed");
  TRY(fi->engine->set_ext_wrench_device(shard, w));
}
/* per-environment mass properties of declared links (Engine::set_mass_prop): an input held like the external wrench */
extern "C" int rkFDBatchSetMassPropLinks(rkFD *fd, int n, const int *links)
{
  BATCH_GUARD(fd);
  if( fi->engine ) return fail("rkFDBatchSetMassPropLinks: declare the links before rkFDUpdateInit");
  if( n < 0 || n > MAX_LINKS ) return fail("rkFDBatchSetMassPropLinks: n must be in [0, " + std::to_string(MAX_LINKS) + "]");
  if( n > 0 && !links ) return fail("rkFDBatchSetMassPropLinks: links is needed");
  const int nl = rkFDBatchLinkNum(fd);
  std::vector<char> seen(nl > 0 ? nl : 1, 0);
  for(int k=0;k<n;k++){
    const int i = links[k];
    if( i < 0 || i >= nl ) return fail("rkFDBatchSetMassPropLinks: link " + std::to_string(i) + " out of range [0, " + std::to_string(nl) + ")");
    if( seen[i] ) return fail("rkFDBatchSetMassPropLinks: link " + std::to_string(i) + " listed twice");
    seen[i] = 1;
  }
  fi->mp_links.assign(links, links + n);
  fi->pend_mp.clear();                /* values held for an earlier declaration have another row count */
  return 0;
}
/* "" when row r = (mass, c, Ic xx xy xz yy yz zz) is physical: finite, mass > 0, Ic positive definite (Cholesky) */
static std::string mass_prop_problem(const double *r)
{
  for(int k=0;k<10;k++) if( !std::isfinite(r[k]) ) return "a non-finite entry";
  if( !( r[0] > 0.0 ) ) return "mass " + std::to_string(r[0]) + " is not positive";
  const double xx = r[4], xy = r[5], xz = r[6], yy = r[7], yz = r[8], zz = r[9];
  if( !( xx > 0.0 ) ) return "the inertia is not positive definite";
  const double l11 = std::sqrt(xx), l21 = xy/l11, l31 = xz/l11, d2 = yy - l21*l21;
  if( !( d2 > 0.0 ) ) return "the inertia is not positive definite";
  const double l22 = std::sqrt(d2), l32 = (yz - l31*l21)/l22, d3 = zz - l31*l31 - l32*l32;
  if( !( d3 > 0.0 ) ) return "the inertia is not positive definite";
  return "";
}
extern "C" int rkFDBatchSetMassProp(rkFD *fd, const double *mp)
{
  BATCH_GUARD(fd);
  if( fi->mp_links.empty() ) return fail("rkFDBatchSetMassProp: no link is declared (rkFDBatchSetMassPropLinks)");
  if( !mp ) return fail("rkFDBatchSetMassProp: mp is needed");
  const size_t n = fi->mp_links.size();
  for(int e=0;e<fi->B;e++) for(size_t k=0;k<n;k++){
    const std::string why = mass_prop_problem(mp + ((size_t)e*n + k)*10);
    if( !why.empty() ) return fail("rkFDBatchSetMassProp: environment " + std::to_string(e) + ", link " + std::to_string(fi->mp_links[k]) + ": " + why);
  }
  if( !fi->engine ){ fi->pend_mp.assign(mp, mp + (size_t)fi->B*10*n); return 0; }
  TRY(fi->engine->set_mass_prop(mp));
}
extern "C" int rkFDBatchSetMassPropDevice(rkFD *fd, int shard, const double *mp)
{
  BATCH_GUARD(fd); NEED_ENGINE();
  if( fi->engine->model().nmp <= 0 ) return fail("rkFDBatchSetMassPropDevice: no link is declared (rkFDBatchSetMassPropLinks)");
  if( shard < 0 || shard >= fi->engine->num_shards() ) return fail("rkFDBatchSetMassPropDevice: shard index out of range");
  if( !mp ) return fail("rkFDBatchSetMassPropDevice: mp is needed");
  TRY(fi->engine->set_mass_prop_device(shard, mp));
}
/* the step-kernel variant a shard launches (Engine::Engine's choice from the model and the RKFD_* tuning variables) */
extern "C" int rkFDBatchKernelVariant(rkFD *fd, int shard, int v[5])
{
  BATCH_GUARD(fd); NEED_ENGINE();
  if( !v ) return fail("rkFDBatchKernelVariant: v is needed");
  TRY(fi->engine->kernel_variant(shard, v));
}
extern "C" const char *rkFDBatchLastError(void){ return g_err.c_str(); }
extern "C" int rkFDBatchDeviceCount(void){ return device_count(); }
extern "C" int rkFDB200MeasureFp64(double *tflops){ try { *tflops = measure_fp64_tflops(); } catch(const std::exception &ex){ return fail(ex.what()); } return 0; }

/* The flattened device model of the last rkFDUpdateInit as text (one "name: numbers" line per table entry, %.17g): what
 * the kernels will see of the registered chains.  Host-side only - it works without a device, because the world is
 * flattened and checked before a device is looked for.  Returns the length needed (excluding the terminator). */
extern "C" int rkFDB200DescribeModel(rkFD *fd, char *buf, int cap)
{
  FDImpl *fi = FI(fd); if( !fi ) return -1;
  const ModelDev &m = fi->model; std::string s; char t[256];
  auto num = [&](double v){ std::snprintf(t, sizeof t, " %.17g", v); s += t; };
  auto arr = [&](const char *name, int idx, const double *v, int n){ std::snprintf(t, sizeof t, "%s[%d]:", name, idx); s += t; for(int i=0;i<n;i++) num(v[i]); s += "\n"; };
  std::snprintf(t, sizeof t, "dims: %d %d %d %d %d %d %d\nprp: %d %d %d %d %.17g %.17g\n", m.nl, m.nq, m.ncell, m.nbox, m.npair, m.nslot, m.nvert,
                m.solver, m.pyramid, m.max_iter, m.integrator, m.dt, m.friction_weight); s += t;
  for(int i=0;i<m.nl;i++){
    const LinkDev &L = m.link[i];
    const double topo[7] = { (double)L.parent, (double)L.jtype, (double)L.mtype, (double)L.ndof, (double)L.qofs, (double)L.cell_begin, (double)L.cell_end };
    arr("link.topo", i, topo, 7); arr("link.Ro", i, L.Ro, 9); arr("link.po", i, L.po, 3);
    const double mp[13] = { L.mass, L.mc[0], L.mc[1], L.mc[2], L.Io[0], L.Io[1], L.Io[2], L.Io[3], L.Io[4], L.Io[5], L.com[0], L.com[1], L.com[2] }; arr("link.mass", i, mp, 13);
    const double jf[9] = { L.stiffness, L.viscosity, L.coulomb, L.sfriction, L.m_tin, L.m_reg, L.m_jm, L.m_min, L.m_max }; arr("link.joint", i, jf, 9);
  }
  for(int i=0;i<m.ncell;i++){ const CellDev &c = m.cell[i]; const double v[5] = { (double)c.link, (double)c.vofs, (double)c.nvert, (double)c.pair_begin, (double)c.pair_end }; arr("cell", i, v, 5); }
  for(int i=0;i<m.nbox;i++){ arr("box.R", i, m.box[i].R, 9); arr("box.p", i, m.box[i].p, 3); arr("box.half", i, m.box[i].half, 3); }
  for(int i=0;i<m.npair;i++){ const PairDev &p = m.pair[i]; const double v[10] = { (double)p.cell, (double)p.box, (double)p.sofs, (double)p.type, p.K, p.L, p.E, p.V, p.SF, p.KF }; arr("pair", i, v, 10); }
  for(int i=0;i<m.nvert;i++) arr("vert", i, m.vert + 3*i, 3);
  /* slide mode: entries (speed, axis, frame of a static box's link) and, per pair that has one, (entry of the vertex's cell + 1, entry
   * of the box + 1, the vertex's cell registered first) */
  for(int i=0;i<m.nslide;i++){ const SlideDev &d = m.slide[i]; double v[16] = { d.vel, d.axis[0], d.axis[1], d.axis[2] };
    for(int k=0;k<9;k++) v[4+k] = d.lR[k]; for(int k=0;k<3;k++) v[13+k] = d.lp[k]; arr("slide", i, v, 16); }
  for(int i=0;i<m.npair;i++) if( m.pair[i].slinfo & 0xffff ){ const int si = m.pair[i].slinfo; const double v[3] = { (double)(si & 255), (double)((si >> 8) & 255), (double)((si >> 16) & 1) }; arr("pair.slide", i, v, 3); }
  /* links declared for an external wrench, in the order of its rows (rkFDBatchSetExtWrenchLinks) */
  if( m.nfext > 0 ){ double v[MAX_LINKS]; for(int i=0;i<m.nl;i++) if( m.link[i].fext_row >= 0 ) v[m.link[i].fext_row] = i; arr("ext.links", 0, v, m.nfext); }
  /* links declared for per-environment mass properties, in the order of their rows (rkFDBatchSetMassPropLinks) */
  if( m.nmp > 0 ){ double v[MAX_LINKS]; for(int i=0;i<m.nl;i++) if( m.mp_row[i] >= 0 ) v[m.mp_row[i]] = i; arr("mp.links", 0, v, m.nmp); }
  if( fd->dis && fd->size > 0 ) arr("init.q", 0, fd->dis->buf, fd->size);     /* the registered initial displacements ([roki::chain::init]) */
  if( buf && cap > 0 ){ std::snprintf(buf, cap, "%s", s.c_str()); }
  return (int)s.size();
}

/* ---- function forms of the reference macros (FFI convenience) ------------------------------------------ */
extern "C" rkFD *rkFDB200Alloc(void){ return (rkFD*)std::calloc(1, sizeof(rkFD)); }
extern "C" void rkFDB200Free(rkFD *fd){ std::free(fd); }
extern "C" rkChain *rkChainB200Alloc(void){ return (rkChain*)std::calloc(1, sizeof(rkChain)); }
extern "C" void rkChainB200Free(rkChain *c){ std::free(c); }
extern "C" void rkFDB200PrpSet(rkFD *fd, double dt, int pyramid, double fw, int max_iter)
{ rkFDPrpSetDT(fd, dt); rkFDPrpSetPyramid(fd, pyramid); rkFDPrpSetFrictionWeight(fd, fw); rkFDPrpSetMaxIter(fd, max_iter); }
extern "C" int rkFDB200SetIntegrator(rkFD *fd, int integrator)      /* function form of rkFDODE2AssignRegular for FFI callers */
{
  if( integrator < RKFD_ODE_RKG || integrator > RKFD_ODE_Heun ) return 1;
  fd->ode.form = RKFD_ODE2_Regular; fd->ode.integrator = integrator; return 0;
}
extern "C" int rkFDB200SetSolver(rkFD *fd, int solver)
{
  if( !FI(fd) ) return 1;
  switch(solver){
    case 0: rkFDSetSolver(fd, Vert); break;
    case 1: rkFDSetSolver(fd, MLCP); break;
    case 2: rkFDSetSolver(fd, Volume); break;
    default: return fail("unknown solver");
  }
  return 0;
}
extern "C" double rkFDB200Time(rkFD *fd){ return rkFDTime(fd); }
extern "C" int rkFDB200Size(rkFD *fd){ return fd->size; }
extern "C" rkChain *rkFDB200CellChain(rkFDCell *cell){ return cell ? rkFDCellChain(cell) : NULL; }
extern "C" const double *rkFDB200Dis(rkFD *fd){ return fd->dis ? fd->dis->buf : NULL; }
extern "C" const double *rkFDB200Vel(rkFD *fd){ return fd->vel ? fd->vel->buf : NULL; }
extern "C" const double *rkFDB200Acc(rkFD *fd){ return fd->acc ? fd->acc->buf : NULL; }
