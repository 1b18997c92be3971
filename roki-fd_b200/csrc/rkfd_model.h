/* rkfd_model.h - host-side chain model (what the reference keeps in rkChain/rkLink/rkJoint/rkMotor,
 * [EXT] RoKi) and its flattening into the constant-memory tables of rkfd_types.h. */
#ifndef RKFD_MODEL_H
#define RKFD_MODEL_H

#include <string>
#include <vector>

#include "rkfd_types.h"

namespace rkfd {

struct MotorHost {
  int type = M_NONE;
  double k = 0, admittance = 0, gear = 1, rotor_inertia = 0, gear_inertia = 0, min = -1e300, max = 1e300;
};

/* zeo box: depth along ax, width along ay, height along az; R = [ax ay az] (columns, row-major storage), identity by default */
struct BoxShape { double center[3]; double depth, width, height; double R[9] = {1,0,0, 0,1,0, 0,0,1};
                  int cloud = -1;   /* moving link: index in LinkHost::shapes of the box's corner cloud (-1: the clouds trail the shapes) */ };

struct LinkHost {
  std::string name, stuff;
  int parent = -1;
  int jtype = J_FIXED;
  double Ro[9] = {1,0,0, 0,1,0, 0,0,1};
  double po[3] = {0,0,0};
  double mass = 0;
  double com[3] = {0,0,0};
  double inertia[9] = {0,0,0, 0,0,0, 0,0,0};
  double stiffness = 0, viscosity = 0, coulomb = 0, sfriction = 0;
  double brk_f = 0, brk_t = 0;               /* breakable float: force / torque thresholds */
  MotorHost motor;
  std::vector<std::vector<double>> shapes;   /* vertex clouds, 3 doubles per vertex, link frame */
  std::vector<BoxShape> boxes;               /* box primitives (kept for static links) */
  /* slide mode per collision cell of the link (rkFDCDCellSetSlideMode/-Vel/-Axis): cell = index among the link's cells (moving
   * link: shapes, then the corner clouds of its boxes; static link: its boxes) */
  struct Slide { int cell; bool mode; double vel; double axis[3]; };
  std::vector<Slide> slides;
  const Slide *slide_of(int cell) const { for(const Slide &s : slides) if( s.cell == cell && s.mode ) return &s; return nullptr; }
};

inline int jtype_ndof(int jt){
  switch(jt){ case J_REVOL: case J_PRISM: return 1; case J_CYLIN: case J_HOOKE: return 2; case J_SPHER: return 3; case J_FLOAT: case J_BRFLOAT: return 6; default: return 0; }
}

struct ChainHost {
  std::string name;
  std::vector<LinkHost> links;
  /* scalar-API mirror of the joint values ([EXT] rkJointGetDis/GetVel/MotorSetInput) */
  std::vector<double> dis, vel, acc, motor_in;
  bool self_collide = true;      /* pairs between the cells of this chain are registered until rkCDPairChainUnreg ([EXT] RoKi rk_cd) */
  int joint_size() const { int n = 0; for(auto &l : links) n += jtype_ndof(l.jtype); return n; }
  bool is_static() const { return joint_size() == 0; }
  int link_qofs(int i) const { int n = 0; for(int k=0;k<i;k++) n += jtype_ndof(links[k].jtype); return n; }
  void sync_sizes(){ int n = joint_size(); dis.resize(n,0.0); vel.resize(n,0.0); acc.resize(n,0.0); motor_in.resize(links.size(),0.0); }
};

struct ContactInfoHost {
  std::string a, b;
  int type = C_RIGID;
  double K = 0, L = 0, E = 0, V = 0, SF = 0, KF = 0;
};

struct WorldHost {
  std::vector<const ChainHost*> chains;     /* registration order */
  std::vector<ContactInfoHost> ci;
  ContactInfoHost cidef;
  double dt = 0.001, friction_weight = 100.0;
  int pyramid = 8, max_iter = 10, solver = S_VERT, integrator = 0;
  std::vector<int> fext_links;              /* links that take an external wrench, in the order of its input rows */
};

/* Flattens the world into `out`.  Returns false and fills `err` when a limit of the fused kernel is
 * exceeded or the topology is not supported. */
bool build_model(const WorldHost &w, ModelDev &out, std::string &err);

/* Scratch map of the generic kernel.  tm = false: everything in the shared-memory column.  tm = true (worlds without
 * rigid pairs): (sin, cos, 1/D, u) of the 1-DoF joints and the integrator stage state move to the T space (tensor
 * memory), the column keeps the rest.  Rewrites slot/sc/wslot/branch/accum/wext/frame slots, rk_slot, nscratch, ntspace. */
void model_layout(ModelDev &m, bool tm);

/* Table of the kinematics pass (rkfd_kin.cuh) for output columns links[0..nlink) (link indices of the model; null: all links,
 * then nlink must be m.nl): the links to visit (the requested ones and their ancestors, parents first), the output columns of
 * each, and the keep slots of frames that a later child needs.  Returns false and fills `err` for a list it refuses
 * (nlink < 0 or > MAX_LINKS, an index out of range). */
bool kin_table(const ModelDev &m, int nlink, const int *links, KinDev &t, std::string &err);

}  // namespace rkfd
#endif
