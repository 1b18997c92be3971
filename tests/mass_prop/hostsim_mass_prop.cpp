/* hostsim_mass_prop.cpp - TEST-ONLY: per-environment mass properties (StateDev::mp) for the host harness of the kernel core.  It
 * compiles tests/hostsim/hostsim.cpp unchanged into its own library and adds entries that work on a HostSim made by
 * libhostsim.so (the same source and flags, so the same layout): the declaration, which flattens the world again and fills
 * the rows with the model's own values, and the rows of every environment. */
#include "../hostsim/hostsim.cpp"

extern "C" {

/* links that take mass properties, in the order of their rows; the model and the state arrays are built again (set the state
 * afterwards, and declare external wrenches before this).  Returns 0 on success */
int hostsim_mp_declare(HostSim *h, int n, const int *links)
{
  h->world.mp_links.assign(links, links + n);
  if( hostsim_finalize(h, h->B) != 0 ) return 1;
  std::vector<double> def; ModelDev *tmp = new ModelDev;
  const bool ok = build_model(h->world, *tmp, h->err, &def);
  delete tmp;
  if( !ok ) return 1;
  const int nr = 10*h->model.nmp, B = h->B;
  h->st.mp = halloc<double>(h, (size_t)(nr > 0 ? nr : 1)*B);
  for(int k=0;k<nr;k++) for(int e=0;e<B;e++) h->st.mp[(size_t)k*B+e] = def[k];
  if( h->spec && h->spec != SPEC_GENERIC_TM && !(spec_match_mask(h->model) >> h->spec & 1u) ) h->spec = 0;
  return 0;
}
/* the mass properties of every environment, env-major mp[B][nmp][10] */
void hostsim_mp_set(HostSim *h, const double *mp)
{
  const int n = 10*h->model.nmp, B = h->B;
  for(int e=0;e<B;e++) for(int k=0;k<n;k++) h->st.mp[(size_t)k*B+e] = mp[(size_t)e*n+k];
}
int hostsim_mp_nmp(HostSim *h){ return h->model.nmp; }

}  // extern "C"
