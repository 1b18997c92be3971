/* ork_ext_wrench.c - TEST-ONLY: the oracle (oracle/rkfd_oracle.c, compiled in unchanged) with external wrenches on links, the
 * reference for rkFDBatchSetExtWrench.  The reference has no such input ([EXT], our convention): per link, a force at the centre
 * of mass and a torque about it, world axes, held like the motor input.  The oracle clears every link's wrench in pass 1 of each
 * evaluation (eval_kinematics: memset of lw[i].wext, after the link's world frame is known); this file routes that clear through
 * a hook which, for the environment being evaluated, sets the wrench to (Rw^T f, Rw^T n + c x Rw^T f) - about the link origin in
 * link axes - instead of zero.  The contact wrenches then add to it, and pass 2 subtracts the sum from the bias, as for contacts.
 * Environments are driven through the ork_ext_* calls below, which name the wrench table W[nl][6] of the environment. */
#include <string.h>
#include <stddef.h>

static void *ork_ext_clear(void *p, int v, size_t n);
#define memset(p, v, n) ork_ext_clear((p), (v), (n))
#include "../../oracle/rkfd_oracle.c"
#undef memset

static __thread ork_env *g_env;          /* environment under evaluation and its wrench table (null: plain oracle) */
static __thread const double *g_w;

static void *ork_ext_clear(void *p, int v, size_t n)
{
  memset(p, v, n);
  if( !g_env || !g_w || n != sizeof g_env->lw[0].wext ) return p;
  for(int i=0;i<g_env->w->nl;i++){
    ork_lw *x = &g_env->lw[i];
    if( p != (void*)x->wext ) continue;
    const double *f = g_w + 6*i; double t[3];
    m3_tmulv(x->Rw,f,x->wext); m3_tmulv(x->Rw,f+3,x->wext+3);
    v3_cross(g_env->w->link[i].com,x->wext,t); v3_add(x->wext+3,t,x->wext+3);
  }
  return p;
}

/* the oracle's calls with the wrench table W[nl][6] of environment e in effect */
void ork_ext_update_init(ork_env *e, const double *W){ g_env = e; g_w = W; ork_env_update_init(e); g_env = NULL; g_w = NULL; }
void ork_ext_update(ork_env *e, const double *W){ g_env = e; g_w = W; ork_env_update(e); g_env = NULL; g_w = NULL; }
void ork_ext_eval(ork_env *e, const double *W, int ref){ g_env = e; g_w = W; ork_env_eval(e, ref); g_env = NULL; g_w = NULL; }
