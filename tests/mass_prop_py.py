"""TEST-ONLY helpers for per-environment mass properties (rkFDBatchSetMassProp): the reference for an environment, the
unchanged oracle on a copy of the world whose declared links carry that environment's mass, centre of mass and inertia, and
the rows the tests set.  The host harness of the kernel core takes the rows itself (hostsim_py.HostSim(..., mp_links=...))."""
import copy

import numpy as np

from oracle.oracle import OracleWorld


def row(mass, com, inertia):
    """(mass, com, Ic xx xy xz yy yz zz): the row of one link"""
    I = np.asarray(inertia, float)
    return np.array([mass, *np.asarray(com, float), I[0, 0], I[0, 1], I[0, 2], I[1, 1], I[1, 2], I[2, 2]])


def own_rows(w, links):
    """(n, 10): the model's own mass properties of `links`"""
    fl = w.flat_links()
    return np.array([row(fl[l].mass, fl[l].com, 0.5 * (np.asarray(fl[l].inertia) + np.asarray(fl[l].inertia).T)) for l in links])


def world_with(w, links, rows):
    """a copy of world w whose links `links` (flat_links() indices) carry the mass properties rows[k]"""
    we = copy.deepcopy(w)
    objs = [l for c in we.moving_chains() for l in c.links]       # the links flat_links() copies, in its order
    for l, r in zip(links, rows):
        o = objs[l]
        o.mass, o.com = float(r[0]), np.array(r[1:4], float)
        o.inertia = np.array([[r[4], r[5], r[6]], [r[5], r[7], r[8]], [r[6], r[8], r[9]]], float)
    return we


def oracle_run_mp(w, q, qd, u, links, MP, nsteps, W=None, wlinks=None):
    """every environment e through the unchanged oracle on world_with(w, links, MP[e]): (q, q', q'') after rkFDUpdateInit and
    nsteps steps.  W (B, len(wlinks), 6): external wrenches on wlinks as well (ext_wrench_py.oracle_run)"""
    out = [np.zeros_like(q), np.zeros_like(q), np.zeros_like(q)]
    for e in range(q.shape[0]):
        we = world_with(w, links, MP[e])
        if W is None:
            r = OracleWorld(we).batch_run(q[e:e + 1], qd[e:e + 1], u[e:e + 1], nsteps=nsteps)
        else:
            from ext_wrench_py import oracle_run
            r = oracle_run(we, q[e:e + 1], qd[e:e + 1], u[e:e + 1], wlinks, W[e:e + 1], nsteps)
        for k in range(3):
            out[k][e] = r[k][0]
    return out


def randomise(w, links, B, seed, mass=0.5, com=0.02, scale=(0.5, 1.5)):
    """(B, n, 10): the model's own values with masses randomised by +-mass, centres of mass shifted by up to `com` and inertias
    scaled by a factor in `scale` (positive definite by construction)"""
    rng = np.random.default_rng(seed)
    base = own_rows(w, links)
    MP = np.repeat(base[None], B, axis=0)
    MP[:, :, 0] *= rng.uniform(1 - mass, 1 + mass, (B, len(links)))
    MP[:, :, 1:4] += rng.uniform(-com, com, (B, len(links), 3))
    MP[:, :, 4:] *= rng.uniform(*scale, (B, len(links), 1))
    return MP
