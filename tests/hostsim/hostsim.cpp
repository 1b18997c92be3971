/* hostsim.cpp - TEST-ONLY host harness: compiles the kernel core (roki-fd_b200/csrc/rkfd_core.cuh)
 * and the link kinematics walk (rkfd_kin.cuh) with g++ and runs them one environment at a time on
 * the CPU, so that the arithmetic of the sm_100a kernels can be checked against the oracle where no
 * GPU exists (`-m "not gpu"` tests).
 * It is NOT part of the product: librokifd_b200.so does not contain it and nothing under
 * roki-fd_b200/ loads it.  The product path has no CPU fallback. */
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#define RKFD_VOL_STATS
static long long rkfd_vol_stats[8];
#include "rkfd_core.cuh"
#include "rkfd_kin.cuh"
#include "rkfd_model.h"

using namespace rkfd;

namespace {
void sincos(double x, double *s, double *c){ *s = std::sin(x); *c = std::cos(x); }
}

struct HostCtx {
  StateDev st; int e, cur; std::vector<double> scr, wsp, tsp; bool tm = false;
  double &S(int k){ return scr[k]; }
  /* T space: a separate array when the specialisation keeps it in tensor memory, the scratch column otherwise */
  double TL(int k){ return tm ? tsp[k] : scr[k]; }
  void TL2(int k, double &a, double &b){ a = TL(k); b = TL(k+1); }
  void TS(int k, double v){ if( tm ) tsp[k] = v; else scr[k] = v; }
  void tfence(){}
  static constexpr bool RIGID = true;
  /* a "warp" of one lane */
  int lanes() const { return 1; }
  int lane() const { return 0; }
  unsigned ballot(bool p) const { return p ? 1u : 0u; }
  bool any(bool p) const { return p; }
  template <class T> T bcast(T x, int) const { return x; }
  double allsum(double x) const { return x; }
  void select(int){}
  void unselect(){}
  void gsync(){}
  void hsync(){}
  bool hany(bool p) const { return p; }
  bool block_or(bool p) const { return p; }
  void phase_sync(int){}
  double &W(int i){ return wsp[i]; }
  double &W1(int i){ return st.ws1[(size_t)i*st.ld + e]; }
  double gld(const double *p, int k) const { return p[(size_t)k*st.ld + e]; }
  void gst(double *p, int k, double v){ p[(size_t)k*st.ld + e] = v; }
};

struct HostSim {
  ModelDev model; WorldHost world; std::vector<ChainHost*> chains; std::string err;
  int B = 0, cur = 0, spec = 0; StateDev st; std::vector<void*> allocs; std::vector<double> last_ws;
};

template <class T> static T *halloc(HostSim *h, size_t n){ void *p = std::calloc(n ? n : 1, sizeof(T)); h->allocs.push_back(p); return (T*)p; }

extern "C" {

/* flat description: same packing as oracle/rkfd_oracle.h (ORK_LINK_ND doubles, 4 ints per link);
 * chain_nl[c] links per chain; stuff ids are turned into names "s<id>" */
HostSim *hostsim_new(int nchain, const int *chain_nl, const int *li, const double *ld)
{
  HostSim *h = new HostSim; int k = 0;
  for(int c=0;c<nchain;c++){
    ChainHost *ch = new ChainHost; ch->name = "chain";
    for(int i=0;i<chain_nl[c];i++,k++){
      LinkHost l; const double *d = ld + 37*k;
      l.parent = li[4*k]; l.jtype = li[4*k+1]; l.motor.type = li[4*k+2]; l.stuff = "s" + std::to_string(li[4*k+3]);
      std::memcpy(l.Ro, d, 72); std::memcpy(l.po, d+9, 24); l.mass = d[12]; std::memcpy(l.com, d+13, 24); std::memcpy(l.inertia, d+16, 72);
      l.stiffness = d[25]; l.viscosity = d[26]; l.coulomb = d[27]; l.sfriction = d[28];
      l.motor.k = d[29]; l.motor.admittance = d[30]; l.motor.gear = d[31]; l.motor.rotor_inertia = d[32];
      l.motor.gear_inertia = d[33]; l.motor.min = d[34]; l.motor.max = d[35];
      if( l.jtype == J_BRFLOAT ){ l.brk_f = d[36]; l.brk_t = d[29]; }     /* thresholds ride in spare fields (no motor on such a link) */
      ch->links.push_back(l);
    }
    h->chains.push_back(ch); h->world.chains.push_back(ch);
  }
  h->world.cidef.type = C_RIGID; h->world.cidef.K = 1000.0; h->world.cidef.L = 1.0; h->world.cidef.SF = 0.5; h->world.cidef.KF = 0.3;
  return h;
}
void hostsim_add_cell(HostSim *h, int chain, int link, int nvert, const double *v)
{ h->chains[chain]->links[link].shapes.push_back(std::vector<double>(v, v+3*nvert)); }
void hostsim_add_box(HostSim *h, int chain, int link, const double *center, double d, double w, double ht)
{ BoxShape b; std::memcpy(b.center, center, 24); b.depth = d; b.width = w; b.height = ht; h->chains[chain]->links[link].boxes.push_back(b); }
void hostsim_unreg_self_collision(HostSim *h, int chain){ h->chains[chain]->self_collide = false; }
void hostsim_set_slide(HostSim *h, int chain, int link, int cell, double vel, const double *axis)
{ LinkHost::Slide s; s.cell = cell; s.mode = true; s.vel = vel; std::memcpy(s.axis, axis, sizeof s.axis); h->chains[chain]->links[link].slides.push_back(s); }
void hostsim_add_contact_info(HostSim *h, int sa, int sb, int type, double K, double L, double E, double V, double SF, double KF)
{ ContactInfoHost c; c.a = "s"+std::to_string(sa); c.b = "s"+std::to_string(sb); c.type = type; c.K=K; c.L=L; c.E=E; c.V=V; c.SF=SF; c.KF=KF; h->world.ci.push_back(c); }
void hostsim_set_prp(HostSim *h, double dt, int pyramid, double fw, int max_iter, int solver)
{ h->world.dt = dt; h->world.pyramid = pyramid; h->world.friction_weight = fw; h->world.max_iter = max_iter; h->world.solver = solver;
  if( solver == S_VOLUME ) h->world.cidef.L = 0.001; }
void hostsim_set_integrator(HostSim *h, int integrator){ h->world.integrator = integrator; }
/* links that take per-environment rows, in the order of the rows; kind 0: external wrench, 1: mass properties.  Before
 * hostsim_finalize, which checks the list */
void hostsim_declare(HostSim *h, int kind, int n, const int *links)
{ (kind == 0 ? h->world.fext_links : h->world.mp_links).assign(links, links + n); }

/* returns 0 on success.  As the engine: the external wrenches start at zero and the mass-property rows of every environment
 * with the model's own values */
int hostsim_finalize(HostSim *h, int B)
{
  std::vector<double> def;
  if( !build_model(h->world, h->model, h->err, &def) ) return 1;
  const ModelDev &m = h->model; h->B = B;
  const int nq = m.nq > 0 ? m.nq : 1, nl = m.nl > 0 ? m.nl : 1, ns = m.nslot > 0 ? m.nslot : 1;
  StateDev &st = h->st; std::memset(&st, 0, sizeof st); st.B = B; st.ld = B;
  for(int k=0;k<2;k++){ st.q[k] = halloc<double>(h, (size_t)nq*B); st.qd[k] = halloc<double>(h, (size_t)nq*B); }
  st.qdd = halloc<double>(h, (size_t)nq*B); st.u = halloc<double>(h, (size_t)nl*B); st.piv_prev = halloc<double>(h, (size_t)nq*B);
  st.piv_type = halloc<unsigned int>(h, B); st.cflags = halloc<unsigned long long>(h, (size_t)(m.nfw > 0 ? m.nfw : 1)*B);
  st.ws1 = halloc<double>(h, (size_t)(m.ws1_doubles > 0 ? m.ws1_doubles : 1)*B);
  st.cref = halloc<double>(h, (size_t)3*ns*B); st.cf = halloc<double>(h, (size_t)3*ns*B); st.status = halloc<int>(h, B);
  if( m.nfext > 0 ) st.fext = halloc<double>(h, (size_t)6*m.nfext*B);
  if( m.nmp > 0 ){
    st.mp = halloc<double>(h, (size_t)10*m.nmp*B);
    for(int k=0;k<10*m.nmp;k++) for(int e=0;e<B;e++) st.mp[(size_t)k*B+e] = def[k];
  }
  return 0;
}
const char *hostsim_error(HostSim *h){ return h->err.c_str(); }
int hostsim_nq(HostSim *h){ return h->model.nq; }
int hostsim_nl(HostSim *h){ return h->model.nl; }
/* model specialisation the kernel would pick (0: generic); hostsim_use_spec makes hostsim_run use it and returns the id
 * it took (0 when the model does not match `id`) */
int hostsim_spec_match(HostSim *h, int tm){ return tm == 2 ? spec_match_rolled(h->model) : spec_match(h->model, tm); }   /* 2: rolled */
unsigned hostsim_spec_mask(HostSim *h){ return spec_match_mask(h->model); }
int hostsim_use_spec(HostSim *h, int id){
  if( id == SPEC_GENERIC_TM ) h->spec = h->model.has_rigid ? 0 : id;
  else h->spec = ( id > 0 && (spec_match_mask(h->model) >> id & 1u) ) ? id : 0;
  return h->spec; }
int hostsim_nslot(HostSim *h){ return h->model.nslot; }
int hostsim_nscratch(HostSim *h){ return h->model.nscratch; }
void hostsim_free(HostSim *h){ for(void *p : h->allocs) std::free(p); for(auto *c : h->chains) delete c; delete h; }

void hostsim_set_state(HostSim *h, const double *q, const double *qd, const double *u)
{
  const int nq = h->model.nq, nl = h->model.nl, B = h->B;
  for(int e=0;e<B;e++){
    for(int j=0;j<nq;j++){ h->st.q[h->cur][(size_t)j*B+e] = q[(size_t)e*nq+j]; h->st.qd[h->cur][(size_t)j*B+e] = qd[(size_t)e*nq+j]; }
    if( u ) for(int j=0;j<nl;j++) h->st.u[(size_t)j*B+e] = u[(size_t)e*nl+j];
  }
}
/* the wrench of every environment, env-major w[B][nfext][6]: (force at the centre of mass, torque about it), world axes */
void hostsim_ext_set(HostSim *h, const double *w)
{
  const int n = 6*h->model.nfext, B = h->B;
  for(int e=0;e<B;e++) for(int k=0;k<n;k++) h->st.fext[(size_t)k*B+e] = w[(size_t)e*n+k];
}
int hostsim_ext_nfext(HostSim *h){ return h->model.nfext; }
/* the mass properties of every environment, env-major mp[B][nmp][10] */
void hostsim_mp_set(HostSim *h, const double *mp)
{
  const int n = 10*h->model.nmp, B = h->B;
  for(int e=0;e<B;e++) for(int k=0;k<n;k++) h->st.mp[(size_t)k*B+e] = mp[(size_t)e*n+k];
}
int hostsim_mp_nmp(HostSim *h){ return h->model.nmp; }
void hostsim_get_state(HostSim *h, double *q, double *qd, double *qdd)
{
  const int nq = h->model.nq, B = h->B;
  for(int e=0;e<B;e++) for(int j=0;j<nq;j++){
    q[(size_t)e*nq+j] = h->st.q[h->cur][(size_t)j*B+e]; qd[(size_t)e*nq+j] = h->st.qd[h->cur][(size_t)j*B+e];
    qdd[(size_t)e*nq+j] = h->st.qdd[(size_t)j*B+e]; }
}
void hostsim_get_contact(HostSim *h, int *active, int *type, double *ref, double *f)
{
  const ModelDev &m = h->model; const int ns = m.nslot, B = h->B;
  for(int p=0;p<m.npair;p++){ const PairDev &pr = m.pair[p]; const int nv = m.cell[pr.cell].nvert;
    for(int kk=0;kk<nv;kk++){ const int fpos = pr.fofs + kk, k = pr.sofs + kk;
      for(int e=0;e<B;e++){ const unsigned long long wd = h->st.cflags[(size_t)(fpos>>5)*B + e];
        active[(size_t)e*ns+k] = (int)((wd >> (2*(fpos&31))) & 1ull); type[(size_t)e*ns+k] = (int)((wd >> (2*(fpos&31)+1)) & 1ull);
        for(int a=0;a<3;a++){ ref[((size_t)e*ns+k)*3+a] = h->st.cref[(size_t)(3*k+a)*B+e]; f[((size_t)e*ns+k)*3+a] = h->st.cf[(size_t)(3*k+a)*B+e]; } } } }
}
void hostsim_get_pivot(HostSim *h, int *type, double *prev)
{
  const int nq = h->model.nq, B = h->B;
  for(int e=0;e<B;e++) for(int j=0;j<nq;j++){ type[(size_t)e*nq+j] = (h->st.piv_type[e] >> j) & 1u; prev[(size_t)e*nq+j] = h->st.piv_prev[(size_t)j*B+e]; }
}
void hostsim_vol_stats(long long *out, int reset){ for(int i=0;i<8;i++){ out[i] = rkfd_vol_stats[i]; if( reset ) rkfd_vol_stats[i] = 0; } }
void hostsim_get_status(HostSim *h, int *status){ for(int e=0;e<h->B;e++) status[e] = h->st.status[e]; }
/* mode 0: nsteps steps; 1: eval; 2: committing eval */
void hostsim_run(HostSim *h, int mode, int nsteps)
{
  for(int e=0;e<h->B;e++){
    HostCtx ctx; ctx.st = h->st; ctx.e = e; ctx.cur = h->cur; ctx.wsp.assign(h->model.ws_doubles + 1, 0.0);
    ctx.scr.assign((h->spec ? spec_nscratch(h->spec) : h->model.nscratch) + 1, std::nan(""));   /* read-before-write shows up as NaN */
    switch(h->spec){
#define RKFD_SPEC_X(id, nl, cls, tmv) case id: { ctx.tm = tmv != 0; ctx.tsp.assign(spec_ntspace(id) + 1, std::nan("")); Core<HostCtx, SpecOf<id>::type> core(ctx); core.run(h->model, mode, nsteps); } break;
    RKFD_SPEC_TABLE(RKFD_SPEC_X)
#undef RKFD_SPEC_X
#define RKFD_SPEC_X(id, nl, rg, gen) case id: { ctx.tm = true; ctx.tsp.assign(spec_ntspace(id) + 1, std::nan("")); Core<HostCtx, SpecOf<id>::type> core(ctx); core.run(h->model, mode, nsteps); } break;
    RKFD_SPEC_ROLLED_TABLE(RKFD_SPEC_X)
#undef RKFD_SPEC_X
    case SPEC_GENERIC_TM: {     /* the generic core on the tensor-memory scratch map */
      ModelDev mt = h->model; model_layout(mt, true);
      ctx.tm = true; ctx.tsp.assign(mt.ntspace + 1, std::nan("")); ctx.scr.assign(mt.nscratch + 1, std::nan(""));
      Core<HostCtx, SpecGenericTM> core(ctx); core.run(mt, mode, nsteps); } break;
    default: { Core<HostCtx> core(ctx); core.run(h->model, mode, nsteps); } break;
    }
    h->last_ws = ctx.wsp;
  }
  if( mode == 0 && (nsteps & 1) ) h->cur ^= 1;
}

/* the kinematics walk of rkFDBatchGetLinkFrames on the model: frames [B][nlink][12] and velocities [B][nlink][6] (either may
 * be null) of links[0..nlink) (null: all) at the env-major states q, qd [B][nq] and pivot words piv [B] (null: none broken).
 * B is the caller's, not the harness's.  Returns 1 when kin_table refuses the list. */
int hostsim_link_frames(HostSim *h, int B, const double *q, const double *qd, const unsigned *piv, int nlink, const int *links,
                        double *frame, double *vel)
{
  KinDev t;
  if( !kin_table(h->model, nlink, links, t, h->err) ) return 1;
  const int nq = h->model.nq;
  struct Row {
    const double *qr, *qdr; unsigned pv;
    double q(int k) const { return qr[k]; }
    double qd(int k) const { return qdr[k]; }
    unsigned piv() const { return pv; }
  };
  struct Keep {
    std::vector<double> v;
    double ld(int s, int c) const { return v[(size_t)s*KIN_KEEP + c]; }
    void st(int s, int c, double x){ v[(size_t)s*KIN_KEEP + c] = x; }
  };
  struct Out {
    double *f, *v;
    void frame(int k, int c, double x){ f[12*k + c] = x; }
    void vel(int k, int c, double x){ v[6*k + c] = x; }
  };
  for(int e=0;e<B;e++){
    const Row S{q + (size_t)e*nq, qd + (size_t)e*nq, piv ? piv[e] : 0u};
    Keep K; K.v.assign((size_t)KIN_KEEP*(t.nkeep + 1), std::nan(""));     /* read-before-write shows up as NaN */
    Out O{frame ? frame + (size_t)e*12*nlink : nullptr, vel ? vel + (size_t)e*6*nlink : nullptr};
    kin_walk(t, S, K, O, frame != nullptr, vel != nullptr);
  }
  return 0;
}

/* debugging aid: the rigid-contact workspace of the last environment processed */
int hostsim_get_ws(HostSim *h, double *out, int cap, int *offs){ int n = (int)h->last_ws.size(); if( n > cap ) n = cap; for(int i=0;i<n;i++) out[i] = h->last_ws[i];
  offs[0]=h->model.ws_geo; offs[1]=h->model.ws_b; offs[2]=h->model.ws_f; offs[3]=h->model.ws_A; offs[4]=h->model.ws_du; offs[5]=h->model.ws_da; offs[6]=h->model.ws_qp; return n; }

}  // extern "C"
