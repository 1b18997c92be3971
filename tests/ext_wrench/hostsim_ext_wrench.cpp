/* hostsim_ext_wrench.cpp - TEST-ONLY: external wrenches (StateDev::fext) for the host harness of the kernel core.  It compiles
 * tests/hostsim/hostsim.cpp unchanged into its own library and adds two entries that work on a HostSim made by libhostsim.so
 * (the same source and flags, so the same layout): the declaration, which flattens the world again, and the wrench rows. */
#include "../hostsim/hostsim.cpp"

extern "C" {

/* links that take an external wrench, in the order of its rows; the model and the state arrays are built again (set the state
 * afterwards).  Returns 0 on success */
int hostsim_ext_declare(HostSim *h, int n, const int *links)
{
  h->world.fext_links.assign(links, links + n);
  if( hostsim_finalize(h, h->B) != 0 ) return 1;
  if( h->spec && h->spec != SPEC_GENERIC_TM && !(spec_match_mask(h->model) >> h->spec & 1u) ) h->spec = 0;
  return 0;
}
/* the wrench of every environment, env-major w[B][nfext][6]: (force at the centre of mass, torque about it), world axes */
void hostsim_ext_set(HostSim *h, const double *w)
{
  const int n = 6*h->model.nfext, B = h->B;
  if( !h->st.fext ) h->st.fext = halloc<double>(h, (size_t)(n > 0 ? n : 1)*B);
  for(int e=0;e<B;e++) for(int k=0;k<n;k++) h->st.fext[(size_t)k*B+e] = w[(size_t)e*n+k];
}
int hostsim_ext_nfext(HostSim *h){ return h->model.nfext; }

}  // extern "C"
