/* kin_harness.cpp - TEST-ONLY host harness of the link kinematics pass (rkFDBatchGetLinkFrames): compiles the walk of
 * roki-fd_b200/csrc/rkfd_kin.cuh and the table builder kin_table (rkfd_model.cpp) with g++ and runs them one environment at a
 * time on the CPU, so that the arithmetic of rkfd_link_frames_kernel is checked against the oracle where no GPU exists.
 * It is NOT part of the product: librokifd_b200.so does not contain it and nothing under roki-fd_b200/ loads it. */
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

/* sincos: the GNU extension of <math.h> (g++ defines _GNU_SOURCE) */
#include "rkfd_kin.cuh"
#include "rkfd_model.h"

using namespace rkfd;

struct KinHarness { ModelDev model; std::vector<ChainHost*> chains; std::string err; };

extern "C" {

/* flat description: the packing of oracle/rkfd_oracle.h (37 doubles, 4 ints per link), chain_nl[c] links per chain with
 * chain-local parents - as tests/hostsim/hostsim.cpp reads it.  Only the link frames matter here: no cells, no contacts. */
KinHarness *kin_new(int nchain, const int *chain_nl, const int *li, const double *ld)
{
  KinHarness *h = new KinHarness; WorldHost w; int k = 0;
  for(int c=0;c<nchain;c++){
    ChainHost *ch = new ChainHost; ch->name = "chain";
    for(int i=0;i<chain_nl[c];i++,k++){
      LinkHost l; const double *d = ld + 37*k;
      l.parent = li[4*k]; l.jtype = li[4*k+1]; l.stuff = "s" + std::to_string(li[4*k+3]);
      std::memcpy(l.Ro, d, 72); std::memcpy(l.po, d+9, 24); l.mass = d[12]; std::memcpy(l.com, d+13, 24); std::memcpy(l.inertia, d+16, 72);
      ch->links.push_back(l);
    }
    h->chains.push_back(ch); w.chains.push_back(ch);
  }
  if( !build_model(w, h->model, h->err) ) h->model.nl = -1;
  return h;
}
const char *kin_error(KinHarness *h){ return h->err.c_str(); }
int kin_nl(KinHarness *h){ return h->model.nl; }
int kin_nq(KinHarness *h){ return h->model.nq; }
void kin_free(KinHarness *h){ for(auto *c : h->chains) delete c; delete h; }

/* frames [B][nlink][12] and velocities [B][nlink][6] (either may be null) of links[0..nlink) (null: all) at the env-major
 * states q, qd [B][nq] and pivot words piv [B] (null: none broken).  Returns 1 when kin_table refuses the list. */
int kin_frames(KinHarness *h, int B, const double *q, const double *qd, const unsigned *piv, int nlink, const int *links,
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

}  // extern "C"
