/* ork_link_wrench.c - TEST-ONLY: the oracle (oracle/rkfd_oracle.c, compiled in unchanged) with one more call, the reference for
 * rkFDBatchGetLinkContactWrench.  The oracle sums every contact wrench of an evaluation into its link's ork_lw::wext (link
 * frame, about the link origin; it holds nothing else without an external wrench).  ork_env_get_link_wrench returns that sum of
 * the last evaluation in world axes: w[nl][6] = (Rw f, Rw n). */
#include "../../oracle/rkfd_oracle.c"

void ork_env_get_link_wrench(const ork_env *e, double *w)
{
  for(int i=0;i<e->w->nl;i++){
    const ork_lw *x = &e->lw[i];
    m3_mulv(x->Rw, x->wext, w + 6*i); m3_mulv(x->Rw, x->wext + 3, w + 6*i + 3);
  }
}
