/* hostsim_link_contact.cpp - TEST-ONLY: the readout of rkFDBatchGetLinkContactWrench (roki-fd_b200/csrc/rkfd_link_contact.cuh)
 * compiled with g++, next to the host harness of the kernel core (tests/hostsim/hostsim.cpp, compiled in unchanged, so that the
 * walk, the table builder and the model are the ones the harness runs).  The entry takes the model of a harness made by
 * libhostsim.so: this library is built from the same source with the same flags, so HostSim has the same layout in both. */
#include <cstdio>

#include "../hostsim/hostsim.cpp"
#include "rkfd_link_contact.cuh"

extern "C" {

/* w [B][nlink][6] of links[0..nlink) (null: all) at the env-major committed states q [B][nq], pivot words piv [B] and contact
 * forces cf [B][nslot][3] of the harness's model.  Returns 1 when link_contact_table refuses the list; err gets the reason */
int hostsim_link_contact(const HostSim *h, int B, const double *q, const unsigned *piv, const double *cf, int nlink,
                         const int *links, double *w, char *err, int errcap)
{
  LcwDev t; std::string msg;
  if( !link_contact_table(h->model, nlink, links, t, msg) ){ std::snprintf(err, errcap, "%s", msg.c_str()); return 1; }
  const int nq = h->model.nq, ns = h->model.nslot;
  struct Row {
    const double *qr; unsigned pv;
    double q(int k) const { return qr[k]; }
    double qd(int) const { return std::nan(""); }      /* velocities are not walked */
    unsigned piv() const { return pv; }
  };
  struct Keep {
    std::vector<double> v;
    double ld(int s, int c) const { return v[(size_t)s*KIN_KEEP + c]; }
    void st(int s, int c, double x){ v[(size_t)s*KIN_KEEP + c] = x; }
  };
  struct Fr {
    std::vector<double> f;
    void frame(int k, int c, double x){ f[12*k + c] = x; }
    void vel(int, int, double){}
    double fr(int k, int c) const { return f[12*k + c]; }
  };
  struct Cf { const double *r; double f(int s, int a) const { return r[3*s + a]; } };
  struct Out { double *o; double &w(int k, int c){ return o[6*k + c]; } };
  for(int e=0;e<B;e++){
    const Row S{q + (size_t)e*nq, piv ? piv[e] : 0u};
    Keep K; K.v.assign((size_t)KIN_KEEP*(t.kin.nkeep + 1), std::nan(""));     /* read-before-write shows up as NaN */
    Fr F; F.f.assign((size_t)12*(t.kin.nsel + 1), std::nan(""));
    kin_walk(t.kin, S, K, F, true, false);
    const Cf C{cf + (size_t)e*3*ns}; Out O{w + (size_t)e*6*nlink};
    link_contact_reduce(t, h->model.vert, F, C, O);
  }
  return 0;
}

}  // extern "C"
