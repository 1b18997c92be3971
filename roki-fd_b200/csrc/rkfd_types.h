/* rkfd_types.h - plain-data tables shared by the host engine and the sm_100a kernels.
 *
 * One `ModelDev` describes what every environment has in common (the registered chains flattened
 * into a forest of links, collision vertex clouds, static boxes, contact pairs, properties).  It
 * lives in __constant__ memory: all threads of a warp read the same entry, so the constant cache
 * broadcasts it and most entries are consumed directly as DFMA operands.
 * Reference data model: rkFD / rkFDCellDat (reference include/roki_fd/rkfd_sim.h:24-52),
 * rkFDPrp (rkfd_property.h:15-22).
 */
#ifndef RKFD_TYPES_H
#define RKFD_TYPES_H

#include <stdint.h>

namespace rkfd {

/* sized for the reference's largest model (example/model/mighty.ztk: 25 links, 26 DoF, 19 shapes, 701 collision vertices)
 * on a floor; the whole table is ~45 KB of the 64 KB constant bank */
constexpr int MAX_LINKS = 32;
constexpr int MAX_CELLS = 32;
constexpr int MAX_VERTS = 768;
constexpr int MAX_BOXES = 8;
constexpr int MAX_MBOXES = 16;     /* box primitives on moving links: collision targets for the vertices of other links' cells */
constexpr int MAX_PAIRS = 64;
constexpr int MAX_SLOTS = 1024;    /* contact slots per env = sum over (cell, box) pairs of the cell's vertices */
/* Contact flags: 2 bits per slot (active, kinetic) in 64-bit words of 32 slots.  Worlds with at most 32 slots keep them in
 * ONE word (flag position = slot); larger worlds give every pair its own word(s) (PairDev::fofs is a multiple of 32), and
 * the kernel holds one word at a time in a register (Core::flag_select). */
constexpr int MAX_FWORDS = 64;
constexpr int RIGID_MAX_SLOTS = 32; /* the rigid VERTEX solvers (MLCP, Vert) address every rigid slot through one flag word */
constexpr int MAX_PYRAMID = 16;

enum JointType : int { J_FIXED = 0, J_REVOL = 1, J_PRISM = 2, J_SPHER = 3, J_FLOAT = 4,
                       J_CYLIN = 5,      /* [EXT] cylindrical: (translation along z, rotation about z) */
                       J_HOOKE = 6,      /* [EXT] hooke / universal: R = Rz(q0) Ry(q1) */
                       J_BRFLOAT = 7 };  /* [EXT A-17] breakable float: rigid until the wrench it transmits exceeds a threshold in a committing
                                          * evaluation, a float joint from then on (pivot bit of its first dof = broken) */
enum MotorType : int { M_NONE = 0, M_DC = 1, M_TRQ = 2 };
enum ContactType : int { C_RIGID = 0, C_ELASTIC = 1 };
enum FricType : int { F_SF = 0, F_KF = 1 };
enum SolverType : int { S_VERT = 0, S_MLCP = 1, S_VOLUME = 2 };

constexpr double GRAVITY = 9.80665;   /* RoKi RK_G */
constexpr double ZTOL = 1.0e-12;      /* ZM zTOL */

struct LinkDev {
  double Ro[9];        /* org frame rotation w.r.t. parent, row-major */
  double po[3];        /* org frame position */
  double pol[3];       /* Ro^T po */
  int rcls;            /* RoClass of Ro (rkfd_math.cuh): 0 general, 1 identity, 2/3 quarter turn about x */
  int fext_row;        /* >=0: row of this link's external wrench in StateDev::fext (rkFDBatchSetExtWrenchLinks), else -1.  It
                          fills the alignment gap before rsg, so no other entry of the table moves */
  double rsg;          /* +1 for Rx(+90), -1 for Rx(-90), 0 otherwise (sign read at run time by the rolled specialisation) */
  double mass;
  double com[3];
  double mc[3];        /* mass * com */
  double Io[6];        /* inertia about the link origin (xx,xy,xz,yy,yz,zz) = Ic - m [c x]^2 */
  double stiffness, viscosity, coulomb, sfriction;
  double m_tin;        /* gear*k*admittance  (input torque per volt) */
  double m_reg;        /* (gear*k)^2*admittance (back-EMF resistance per rad/s) */
  double m_jm;         /* gear^2*(rotor+gear inertia) */
  double m_min, m_max;
  int parent, jtype, mtype, ndof, qofs;
  int slot;            /* first scratch slot of this link */
  int sc;              /* 1-DoF joints: index of (sin, cos, 1/D, u) - slot + 6 in the scratch column, or a T-space index in the
                          tensor-memory layout of the generic kernel (model_layout_tm) */
  int wslot;           /* slots of (w, gravity direction) written by pass 1: aliased with U (= slot) unless the world has
                          rigid pairs, where pass 2 runs twice per evaluation and they must survive */
  int serial;          /* 1: parent == index-1 and the parent has no other child (carry in registers) */
  int nchild;          /* number of children */
  int branch_slot;     /* >=0: slots where this link publishes frame/velocity/acceleration for non-serial children */
  int accum_slot;      /* >=0: slots where non-serial children accumulate articulated inertia/bias (27) */
  int wext_slot;       /* >=0: slots of the external wrench (6) (links that carry collision cells or take a wrench, fext_row) */
  int frame_slot;      /* >=0 (worlds with rigid pairs, links with cells): Rw(9) pw(3) vl(3) w(3) a(6) = 24 slots */
  int cell_begin, cell_end;
  double brk_f, brk_t; /* breakable float: force / torque thresholds */
  int mcol;            /* 1: a cell or a box of this link takes part in a moving-vs-moving pair (frame + wrench slots) */
  int pz;              /* 1: revolute / fixed joint whose org position is (0, 0, z): the structured shifts of rkfd_math.cuh apply */
};

struct CellDev { int link, vofs, nvert, pair_begin, pair_end; };
struct BoxDev { double R[9], p[3], half[3]; double lR[9]; };     /* world frame of the box; lR: world rotation of the (static) link that carries it (slide mode) */
struct MBoxDev { double R[9], p[3], half[3]; int link, pad_; };      /* frame in the carrying link */
/* slide mode of a collision cell ("fake crawler", reference rkfd_sim.c:386-440): belt speed, axis in the frame of the cell's link;
 * (lR, lp): world frame of the link of a STATIC box */
struct SlideDev { double vel, axis[3], lR[9], lp[3]; };
constexpr int MAX_SLIDES = 8;
/* slinfo: bits 0-7 = 1 + slide entry of the vertex's cell (0: none), bits 8-15 = the same for the box, bit 16 = the vertex's
 * cell was registered before the box's (it is pd->cell[0], rkFDUpdateRefSlide rkfd_util.c:218-237) */
struct PairDev { int cell, box, sofs, type; double K, L, E, V, SF, KF; int fofs, volbox; int mbox, slinfo; };   /* fofs: flag position of vertex 0 (word fofs>>5, bit pair fofs&31); volbox: the cell has the 8 corners of a box in sign-bit order (Volume solver);
                                 * mbox >= 0: the target is box `mbox` on a moving link (then box = -1): elastic pairs only */

struct ModelDev {
  int nl, nq, ncell, nbox, npair, nslot, nvert;
  int nfw;             /* contact flag words per environment */
  int npair_static;    /* pairs [0, npair_static): against static boxes (walked link by link in pass 1); the rest: against boxes on
                          moving links (walked after pass 1, Core::contacts_moving) */
  int nmbox;
  int need_world;      /* any collision cell: world frames must be propagated */
  int has_rigid, has_elastic;
  int nslide; SlideDev slide[MAX_SLIDES];
  int rigid_moving;    /* a rigid pair of two moving links exists: the dense rigid path (A couples the two links / chains) */
  int solver, pyramid, max_iter;
  int integrator;      /* 0 Runge-Kutta-Gill, 1 classical Runge-Kutta, 2 Euler, 3 Heun ([EXT] zODE2AssignRegular) */
  int nfext;           /* links declared for an external wrench (LinkDev::fext_row); in the alignment gap before rk */
  /* stage coefficients of the integrator times dt, folded on the host (constant-bank operands in the kernel) */
  struct RK { double c21, c31, c32, c42, c43, b1, b2, b3, b4; int ns; } rk;
  int nscratch;        /* scratch slots (doubles) per env */
  int ntspace;         /* tensor-memory layout: T-space doubles per env (per-joint scalars + integrator state), else 0 */
  int ws_doubles;      /* per-warp workspace (doubles) of the rigid-contact solve, 0 when no rigid pair */
  int ws_geo, ws_b, ws_f, ws_A, ws_du, ws_da, ws_qp;   /* offsets inside the workspace */
  int nmax;            /* 3 * (rigid contact slots) */
  int rigid_link;      /* >= 0: the wrench-coordinate contact paths apply (= rg_link[0]); -1: the dense path */
  int nrg, rg_link[4]; /* contact groups of those paths: the links that carry rigid cells, each in a different chain (no dynamic
                          coupling between groups: the reference zeroes those blocks of A, rkfd_vert.c:133-137) */
  int ws1_doubles;     /* per-ENVIRONMENT workspace (doubles) of the single-link MLCP path, 0 when unused */
  unsigned long long rigid_mask;   /* bit 2s set when slot s belongs to a rigid pair */
  int slot_pair[RIGID_MAX_SLOTS], slot_vert[RIGID_MAX_SLOTS];   /* single-word worlds (the rigid vertex solvers) */
  int rk_slot;         /* first slot of the RKG stage state: QS[nq], QDS[nq], PQ[nq], PQD[nq] */
  double dt, friction_weight;
  double inv_dt;       /* 1/dt */
  double sc_sin[MAX_PYRAMID], sc_cos[MAX_PYRAMID];
  double tay[6];       /* Taylor coefficients of Core::rot_sincos as constant-bank operands (a 64-bit literal costs two moves per use) */
  LinkDev link[MAX_LINKS];
  CellDev cell[MAX_CELLS];
  BoxDev box[MAX_BOXES];
  MBoxDev mbox[MAX_MBOXES];
  PairDev pair[MAX_PAIRS];
  double vert[3 * MAX_VERTS];
  /* per-environment mass properties (rkFDBatchSetMassPropLinks), appended so that no entry above moves */
  int nmp;             /* links declared for per-environment mass properties */
  int mp_row[MAX_LINKS];   /* >=0: row of link i's mass properties in StateDev::mp, else -1 */
};

/* Link table of the kinematics pass (rkfd_kin.cuh, rkFDBatchGetLinkFrames).  It is a __grid_constant__ kernel parameter, not
 * the __constant__ bank of the step kernels (engines share those banks, g_model_owner), and holds what the walk needs: the
 * joint model of every link and which links to visit and report.  ~4.5 KB at MAX_LINKS: within the 32 KB parameter limit. */
struct KinLinkDev {
  double Ro[9], po[3];  /* org frame w.r.t. the parent (LinkDev::Ro, po) */
  double sg;            /* sign of the quarter turn (cls RO_RXP / RO_RXM) */
  int cls, pz, parent, jtype, qofs;
  int keep;             /* >= 0: shared-memory slot where the walk keeps this link's frame for a later child that is not the next
                           link visited; -1: the next visited link continues from registers or nothing needs it */
  unsigned omask;       /* bit k: output column k reports this link (duplicates in the list set several bits) */
  int pad_;
};
struct KinDev {
  int nwalk;            /* links visited: the requested links and their ancestors, parents first */
  int nsel;             /* output columns (requested links, duplicates included) */
  int nkeep;            /* shared-memory slots of kept frames (KIN_KEEP doubles each) */
  int brk;              /* the world has breakable-float joints: the kernel reads piv_type */
  int walk[MAX_LINKS];
  KinLinkDev link[MAX_LINKS];   /* indexed by the model's link index */
};
constexpr int KIN_KEEP = 18;    /* Rw (9), pw (3), linear and angular velocity in link axes (3 + 3) */

/* Contact table of the link contact-wrench readout (rkfd_link_contact.cuh, rkFDBatchGetLinkContactWrench): a __grid_constant__
 * kernel parameter like KinDev, ~12 KB at the limits.  `kin` walks the links whose frames the readout needs (its output columns
 * are "frame columns"): the requested links that carry cells or boxes in a pair, and the vertex-side links of moving pairs whose
 * box sits on a requested link.  A term is one (pair, side) that pushes a wrench onto a requested link. */
struct LcwBoxDev {
  double R[9], p[3], half[3];   /* static box: world frame; box on a moving link: frame in that link (MBoxDev) */
  int col;                      /* frame column of the carrying link, -1: static box */
  int pad_;
};
enum LcwKind : int { LCW_VERT = 0,   /* vertex slots of a cell on the link: +f at the vertex */
                     LCW_BOX = 1,    /* box of a moving pair on the link: -f at the vertex of the other link */
                     LCW_VOL = 2 };  /* Volume box pair: slots (force, torque about the centre, centre) */
struct LcwTermDev { int kind, elastic, sofs, vofs, nvert, vcol, box, acc; };   /* acc: output column that accumulates */
constexpr int LCW_MAX_TERMS = 2*MAX_PAIRS;    /* a pair acts on at most two links */
struct LcwDev {
  KinDev kin;
  int nsel;                     /* output columns (requested links, duplicates included) */
  int nterm;
  int first[MAX_LINKS];         /* output column k repeats column first[k] (== k: its own accumulator) */
  int ocol[MAX_LINKS];          /* frame column of the link of output column k (the torque's reference point), -1: no term */
  LcwBoxDev box[MAX_BOXES + MAX_MBOXES];   /* static boxes, then the boxes of moving links */
  LcwTermDev term[LCW_MAX_TERMS];
};

/* Per-environment state in HBM, structure-of-arrays with the environment index fastest:
 * element (k, e) of an array lives at base[k*ld + e].  Thread e of a warp therefore reads
 * consecutive 8-byte words: every load/store is one fully coalesced 256-byte request. */
struct StateDevHead {
  int B;               /* environments on this device */
  int ld;              /* leading dimension (B rounded up to 32) */
  double *q[2], *qd[2];   /* double-buffered committed state [nq][ld] */
  double *qdd;            /* [nq][ld] acceleration of the last reference evaluation */
  double *u;              /* [nl][ld] motor input per link */
  double *piv_prev;       /* [nq][ld] previous driving torque per dof */
  unsigned int *piv_type; /* [ld] bit j: dof j pivot is kinetic   (nq <= 32) */
  unsigned long long *cflags; /* [nfw][ld] 2 bits per flag position: bit 2f active, bit 2f+1 kinetic */
  double *cref;           /* [nslot*3][ld] anchor _ref in the box frame */
  double *cf;             /* [nslot*3][ld] contact force (world) of the last reference evaluation */
  double *scratch;        /* optional global scratch [nscratch][ld] when shared memory is too small */
  double *ws;             /* rigid-contact workspace, ws_doubles per warp (ld/32 warps) */
  double *ws1;            /* [ws1_doubles][ld] per-environment workspace of the single-link MLCP path */
  int *status;            /* [ld] per-env status word (bit0: non-finite acceleration) */
  unsigned char *work;    /* [ld] or null: work class of the environment's last rigid solve (Vert / Volume: pairs or contacts and
                           * active-set iterations), 0 = no solve; the engine's re-sort groups equal classes into warps */
};
/* The step kernel takes the head as its first parameter and fext and mp as its last ones (rkfd_kernel.cuh): its other
 * parameters keep their places in the parameter space, and kernels that never read them compile to the code they had without them */
struct StateDev : StateDevHead {
  double *fext;           /* [6*nfext][ld] or null: external wrench per declared link, (force, torque about the centre of mass),
                           * world axes (row 6*LinkDev::fext_row + k) */
  double *mp;             /* [10*nmp][ld] or null: mass properties per declared link, (mass, centre of mass, inertia about the centre
                           * of mass xx xy xz yy yz zz), link axes (row 10*ModelDev::mp_row[i] + k) */
};

}  // namespace rkfd
#endif
