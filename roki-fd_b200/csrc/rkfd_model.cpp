/* rkfd_model.cpp - flattening of registered chains into the device tables (host only). */
#include "rkfd_model.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>

#include "rkfd_core.cuh"

namespace rkfd {

static void mat3_mul(const double *a, const double *b, double *c){
  double t[9];
  for(int i=0;i<3;i++) for(int j=0;j<3;j++){ t[3*i+j] = 0; for(int k=0;k<3;k++) t[3*i+j] += a[3*i+k]*b[3*k+j]; }
  std::memcpy(c, t, sizeof t);
}
static void mat3_mulv(const double *a, const double *x, double *y){
  double t[3];
  for(int i=0;i<3;i++) t[i] = a[3*i]*x[0] + a[3*i+1]*x[1] + a[3*i+2]*x[2];
  std::memcpy(y, t, sizeof t);
}

void model_layout(ModelDev &m, bool tm)
{
  const int nl = m.nl, nq = m.nq;
  int slot = 0, t = 0;
  for(int i=0;i<nl;i++){
    LinkDev &d = m.link[i];
    d.branch_slot = d.accum_slot = d.wext_slot = d.frame_slot = -1;
    d.slot = slot; d.wslot = slot + link_w_offset(d.jtype, m.has_rigid);
    const bool one = d.jtype == J_REVOL || d.jtype == J_PRISM;
    if( tm && one ){ d.sc = t; t += 4; slot += link_slot_count(d.jtype, m.has_rigid) - 4; d.wslot = d.slot + ( m.has_rigid ? 6 : 0 ); }
    else { d.sc = slot + 6; slot += link_slot_count(d.jtype, m.has_rigid); }
  }
  for(int i=0;i<nl;i++){
    LinkDev &d = m.link[i];
    if( d.parent >= 0 && !d.serial ){
      LinkDev &p = m.link[d.parent];
      if( p.branch_slot < 0 ){ p.branch_slot = slot; slot += BRANCH_SLOTS; p.accum_slot = slot; slot += ACCUM_SLOTS; }
    }
    if( d.cell_end > d.cell_begin || d.mcol || d.fext_row >= 0 ){ d.wext_slot = slot; slot += WEXT_SLOTS;
      /* a link that only takes an external wrench gets no frame slot: the contact paths read frames of links with cells */
      if( ( m.has_rigid && d.cell_end > d.cell_begin ) || d.mcol ){ d.frame_slot = slot; slot += FRAME_SLOTS; } }
  }
  if( tm ){ m.rk_slot = t; t += 4*nq; m.ntspace = t; }
  else { m.rk_slot = slot; slot += 4*nq; m.ntspace = 0; }
  m.nscratch = slot;
}

/* [EXT A-15] vertices of an 8-corner cell into sign-bit order: vertex k = v0 + (k&1) ea + (k>>1&1) eb + (k>>2&1) ec with v0 the
 * first vertex and (a,b,c) the first index triple in lexicographic order that spans the cell, so that polyhedron-described
 * boxes (mighty.ztk's soles: bottom ring, top ring) are accepted; false when the points are not a parallelepiped. */
static bool box_sign_bit_order(double *v)
{
  double scale = 0, out[24];
  for(int k=1;k<8;k++) for(int i=0;i<3;i++) scale = std::max(scale, std::fabs(v[3*k+i]-v[i]));
  const double tol = 1e-9*(1+scale);
  for(int a=1;a<8;a++) for(int b=a+1;b<8;b++) for(int c=b+1;c<8;c++){
    unsigned used = 0; bool ok = true;
    for(int k=0;k<8 && ok;k++){
      double p[3]; int found = -1;
      for(int i=0;i<3;i++) p[i] = v[i] + ((k&1)?v[3*a+i]-v[i]:0.0) + ((k&2)?v[3*b+i]-v[i]:0.0) + ((k&4)?v[3*c+i]-v[i]:0.0);
      for(int j=0;j<8;j++) if( !(used>>j & 1u) && std::fabs(v[3*j]-p[0]) <= tol && std::fabs(v[3*j+1]-p[1]) <= tol && std::fabs(v[3*j+2]-p[2]) <= tol ){ found = j; break; }
      if( found < 0 ){ ok = false; break; }
      used |= 1u<<found; std::memcpy(out+3*k, v+3*found, 24);
    }
    if( ok ){ std::memcpy(v, out, sizeof out); return true; }
  }
  return false;
}

bool build_model(const WorldHost &w, ModelDev &m, std::string &err)
{
  std::memset(&m, 0, sizeof m);
  m.dt = w.dt; m.inv_dt = 1.0/w.dt; m.friction_weight = w.friction_weight; m.pyramid = w.pyramid; m.max_iter = w.max_iter; m.solver = w.solver; m.integrator = w.integrator;
  m.rk = rk_coef(w.dt, w.integrator);
  if( w.pyramid > MAX_PYRAMID || w.pyramid < 1 ){ err = "pyramid order out of range"; return false; }
  m.tay[0] = 1.0/362880.0; m.tay[1] = -1.0/5040.0; m.tay[2] = 1.0/120.0; m.tay[3] = -1.0/6.0; m.tay[4] = 1.0/40320.0; m.tay[5] = -1.0/720.0;
  { /* rkFDCrateSinCosTable (reference rkfd_util.c:199-214) with the Vert offset -pi/pyramid (rkfd_vert.c:369); the Volume
     * solver's table has no offset (rkfd_volume.c:1000) */
    const double off = w.solver == S_VOLUME ? 0.0 : -M_PI / w.pyramid, dth = 2.0*M_PI / w.pyramid; double th = 0.0;
    for(int i=0;i<w.pyramid;i++, th+=dth){ m.sc_sin[i] = std::sin(th+off); m.sc_cos[i] = std::cos(th+off); }
  }

  std::vector<std::string> link_stuff; std::vector<int> link_chain; std::vector<bool> chain_self;
  struct StatBox { BoxDev b; std::string stuff; int ord, slide; };
  std::vector<StatBox> boxes;
  std::vector<int> cell_ord, cell_slide, mbox_ord, mbox_slide;      /* registration order / slide entry (-1: none) of every cell and moving box */
  int ord = 0;                                                       /* shapes in the order of rkFDChainReg: chains, links, shapes then boxes */
  auto add_slide = [&](const LinkHost::Slide *sl, const double *lR, const double *lp) -> int {
    if( !sl ) return -1;
    if( m.nslide >= MAX_SLIDES ) return -2;
    SlideDev &d = m.slide[m.nslide]; d.vel = sl->vel; std::memcpy(d.axis, sl->axis, sizeof d.axis);
    static const double I3[9] = {1,0,0, 0,1,0, 0,0,1}, Z3[3] = {0,0,0};
    std::memcpy(d.lR, lR ? lR : I3, sizeof d.lR); std::memcpy(d.lp, lp ? lp : Z3, sizeof d.lp);
    return m.nslide++; };

  /* ---- moving chains -> forest of links (registration order); static chains -> world boxes */
  int nl = 0, nq = 0;
  for(const ChainHost *ch : w.chains){
    if( ch->is_static() ){
      std::vector<std::vector<double>> fr(ch->links.size(), std::vector<double>(12));
      for(size_t i=0;i<ch->links.size();i++){
        const LinkHost &l = ch->links[i]; double R[9], p[3];
        std::memcpy(R, l.Ro, sizeof R); std::memcpy(p, l.po, sizeof p);
        if( l.parent >= 0 ){
          if( l.parent >= (int)i ){ err = "link order: parent must precede child"; return false; }
          const double *Rp = fr[l.parent].data(), *pp = Rp + 9; double t[3];
          mat3_mul(Rp, l.Ro, R); mat3_mulv(Rp, l.po, t); for(int k=0;k<3;k++) p[k] = pp[k] + t[k];
        }
        std::memcpy(fr[i].data(), R, sizeof R); std::memcpy(fr[i].data()+9, p, sizeof p);
        int bidx = 0;
        for(const BoxShape &bs : l.boxes){
          StatBox sb; double c[3];
          mat3_mul(R, bs.R, sb.b.R); mat3_mulv(R, bs.center, c);
          for(int k=0;k<3;k++) sb.b.p[k] = p[k] + c[k];
          sb.b.half[0] = 0.5*bs.depth; sb.b.half[1] = 0.5*bs.width; sb.b.half[2] = 0.5*bs.height;
          std::memcpy(sb.b.lR, R, sizeof sb.b.lR);
          sb.stuff = l.stuff; sb.ord = ord++; sb.slide = add_slide(l.slide_of(bidx++), R, p);
          if( sb.slide == -2 ){ err = "too many cells in slide mode (MAX_SLIDES)"; return false; }
          boxes.push_back(sb);
        }
      }
      continue;
    }
    const int base = nl;
    chain_self.push_back(ch->self_collide);
    for(size_t i=0;i<ch->links.size();i++){
      const LinkHost &l = ch->links[i];
      if( nl >= MAX_LINKS ){ err = "too many links (MAX_LINKS)"; return false; }
      if( l.parent >= (int)i ){ err = "link order: parent must precede child"; return false; }
      LinkDev &d = m.link[nl];
      d.fext_row = -1;
      std::memcpy(d.Ro, l.Ro, sizeof d.Ro); std::memcpy(d.po, l.po, sizeof d.po);
      d.mass = l.mass;
      for(int k=0;k<3;k++){ d.com[k] = l.com[k]; d.mc[k] = l.mass*l.com[k]; }
      { /* class of the constant rotation; entries within 1e-14 of {0,+-1} are snapped so that the structured
           transforms are exact signed permutations */
        static const double RI[9] = {1,0,0, 0,1,0, 0,0,1}, RP[9] = {1,0,0, 0,0,-1, 0,1,0}, RM[9] = {1,0,0, 0,0,1, 0,-1,0};
        const double *cand[3] = {RI, RP, RM}; d.rcls = RO_GENERAL;
        for(int cidx=0;cidx<3;cidx++){ bool ok = true; for(int k=0;k<9;k++) if( std::fabs(d.Ro[k]-cand[cidx][k]) > 1e-14 ) ok = false;
          if( ok ){ d.rcls = cidx+1; std::memcpy(d.Ro, cand[cidx], sizeof d.Ro); break; } }
        d.rsg = d.rcls == RO_RXP ? 1.0 : ( d.rcls == RO_RXM ? -1.0 : 0.0 );
        for(int k=0;k<3;k++) d.pol[k] = d.Ro[k]*d.po[0] + d.Ro[3+k]*d.po[1] + d.Ro[6+k]*d.po[2];
      }
      { /* Io = Ic - m [c x]^2 = Ic + m (|c|^2 E - c c^T) */
        const double *c = l.com, c2 = c[0]*c[0]+c[1]*c[1]+c[2]*c[2]; double Io[9];
        for(int r=0;r<3;r++) for(int q=0;q<3;q++) Io[3*r+q] = l.inertia[3*r+q] + l.mass*((r==q?c2:0.0) - c[r]*c[q]);
        d.Io[0]=Io[0]; d.Io[1]=0.5*(Io[1]+Io[3]); d.Io[2]=0.5*(Io[2]+Io[6]); d.Io[3]=Io[4]; d.Io[4]=0.5*(Io[5]+Io[7]); d.Io[5]=Io[8];
      }
      d.stiffness = l.stiffness; d.viscosity = l.viscosity; d.coulomb = l.coulomb; d.sfriction = l.sfriction;
      d.brk_f = l.brk_f; d.brk_t = l.brk_t;
      d.mtype = l.motor.type;
      /* [EXT A-6] DC motor constants folded once on the host */
      d.m_tin = l.motor.gear*l.motor.k*l.motor.admittance;
      d.m_reg = (l.motor.gear*l.motor.k)*(l.motor.gear*l.motor.k)*l.motor.admittance;
      d.m_jm  = l.motor.gear*l.motor.gear*(l.motor.rotor_inertia + l.motor.gear_inertia);
      d.m_min = l.motor.min; d.m_max = l.motor.max;
      if( d.mtype == M_TRQ ){ d.m_jm = 0; }
      d.parent = l.parent >= 0 ? l.parent + base : -1;
      d.jtype = l.jtype; d.ndof = jtype_ndof(l.jtype); d.qofs = nq; nq += d.ndof;
      d.pz = ( ( d.jtype == J_REVOL || d.jtype == J_FIXED ) && d.po[0] == 0.0 && d.po[1] == 0.0 ) ? 1 : 0;
      if( d.ndof != 1 ) d.mtype = M_NONE;
      d.cell_begin = m.ncell;
      int cidx = 0;
      for(const auto &sh : l.shapes){
        const int nv = (int)sh.size()/3;
        if( m.ncell >= MAX_CELLS ){ err = "too many collision cells (MAX_CELLS)"; return false; }
        if( m.nvert + nv > MAX_VERTS ){ err = "too many collision vertices (MAX_VERTS)"; return false; }
        CellDev &c = m.cell[m.ncell++]; c.link = nl; c.vofs = m.nvert; c.nvert = nv;
        std::memcpy(m.vert + 3*m.nvert, sh.data(), 3*nv*sizeof(double)); m.nvert += nv;
        /* every cell is one registered shape (a box primitive and its corner cloud are ONE shape of the reference) */
        const int o = ord++;
        const int sl = add_slide(l.slide_of(cidx), nullptr, nullptr);
        if( sl == -2 ){ err = "too many cells in slide mode (MAX_SLIDES)"; return false; }
        cell_ord.push_back(o); cell_slide.push_back(sl); cidx++;
      }
      d.cell_end = m.ncell;
      for(const BoxShape &bs : l.boxes){         /* box primitives of a moving link: targets */
        if( m.nmbox >= MAX_MBOXES ){ err = "too many boxes on moving links (MAX_MBOXES)"; return false; }
        MBoxDev &mb = m.mbox[m.nmbox++]; std::memcpy(mb.R, bs.R, sizeof mb.R); std::memcpy(mb.p, bs.center, sizeof mb.p);
        mb.half[0] = 0.5*bs.depth; mb.half[1] = 0.5*bs.width; mb.half[2] = 0.5*bs.height; mb.link = nl;
        /* its corner cloud is cell `cloud` of the link (recorded by whoever added the box; else the clouds trail the shapes):
         * the box shares registration order and slide entry with it */
        const int k = (int)(&bs - &l.boxes[0]), nshape = (int)l.shapes.size() - (int)l.boxes.size();
        const int cl = bs.cloud >= 0 ? bs.cloud : nshape + k;
        int o = ord, sl = -1;
        if( cl >= 0 && d.cell_begin + cl < (int)cell_ord.size() ){ o = cell_ord[d.cell_begin + cl]; sl = cell_slide[d.cell_begin + cl]; }
        mbox_slide.push_back(sl);
        mbox_ord.push_back(o);
      }
      link_stuff.push_back(l.stuff); link_chain.push_back((int)chain_self.size() - 1);
      nl++;
    }
  }
  m.nl = nl; m.nq = nq;
  if( nq > 32 ){ err = "too many joint dofs for the pivot bitmask (32)"; return false; }
  if( (int)boxes.size() > MAX_BOXES ){ err = "too many static boxes (MAX_BOXES)"; return false; }
  m.nbox = (int)boxes.size();
  for(int b=0;b<m.nbox;b++) m.box[b] = boxes[b].b;

  /* ---- contact pairs (cell x box) with their contact info (reference rkfd_sim.c:200-207, :266-271) */
  int sofs = 0;
  for(int c=0;c<m.ncell;c++){
    m.cell[c].pair_begin = m.npair;
    for(int b=0;b<m.nbox;b++){
      if( m.npair >= MAX_PAIRS ){ err = "too many contact pairs (MAX_PAIRS)"; return false; }
      PairDev &p = m.pair[m.npair++];
      p.cell = c; p.box = b; p.sofs = sofs; sofs += m.cell[c].nvert;
      const ContactInfoHost *ci = &w.cidef;
      const std::string &sa = link_stuff[m.cell[c].link], &sb = boxes[b].stuff;
      for(const auto &e : w.ci) if( (e.a==sa && e.b==sb) || (e.a==sb && e.b==sa) ){ ci = &e; break; }
      p.type = ci->type; p.K = ci->K; p.L = ci->L; p.E = ci->E; p.V = ci->V; p.SF = ci->SF; p.KF = ci->KF;
      if( p.type == C_ELASTIC ) m.has_elastic = 1; else m.has_rigid = 1;
      p.slinfo = (cell_slide[c] + 1) | ((boxes[b].slide + 1) << 8) | ( cell_ord[c] < boxes[b].ord ? 1 << 16 : 0 );
    }
    m.cell[c].pair_end = m.npair;
  }
  for(int p=0;p<m.npair;p++) m.pair[p].mbox = -1;
  m.npair_static = m.npair;
  /* ---- moving-vs-moving pairs ([EXT A-10]: vertices of a cell against a box primitive carried by ANOTHER link - of another
   * chain, or of the same chain while its self-collision pairs are registered, rkCDPairChainUnreg).  Rigid contact info
   * between two moving links goes through the dense vertex solvers (A couples the two links / chains: rkfd_vert.c:125-185,
   * rkfd_mlcp.c:76-142); the Volume solver forms its contact volumes against static boxes only ([EXT A-15]): under it such
   * pairs are left out and reported. */
  { int dropped = 0;
    for(int c=0;c<m.ncell;c++) for(int b=0;b<m.nmbox;b++){
      const int la = m.cell[c].link, lb = m.mbox[b].link;
      if( la == lb ) continue;
      if( link_chain[la] == link_chain[lb] && !chain_self[link_chain[la]] ) continue;
      const ContactInfoHost *ci = &w.cidef;
      const std::string &sa = link_stuff[la], &sb = link_stuff[lb];
      for(const auto &e : w.ci) if( (e.a==sa && e.b==sb) || (e.a==sb && e.b==sa) ){ ci = &e; break; }
      if( ci->type != C_ELASTIC && w.solver == S_VOLUME ){ dropped++; continue; }
      if( m.npair >= MAX_PAIRS ){ err = "too many contact pairs (MAX_PAIRS)"; return false; }
      PairDev &p = m.pair[m.npair++];
      p.cell = c; p.box = -1; p.mbox = b; p.sofs = sofs; sofs += m.cell[c].nvert;
      p.type = ci->type; p.K = ci->K; p.L = ci->L; p.E = ci->E; p.V = ci->V; p.SF = ci->SF; p.KF = ci->KF;
      if( p.type == C_ELASTIC ) m.has_elastic = 1; else { m.has_rigid = 1; m.rigid_moving = 1; }
      p.slinfo = (cell_slide[c] + 1) | ((mbox_slide[b] + 1) << 8) | ( cell_ord[c] < mbox_ord[b] ? 1 << 16 : 0 );
      m.link[la].mcol = 1; m.link[lb].mcol = 1;
    }
    if( dropped ) std::fprintf(stderr, "rokifd_b200: %d pair(s) of cells on two MOVING links have rigid contact info: not formed under the Volume "
                                       "solver (its contact volumes are formed against static boxes)\n", dropped);
  }
  m.nslot = sofs;  /* flag positions: one word when everything fits 32 slots (position = slot), else whole words per pair */
  if( m.nslot <= 32 ){ for(int p=0;p<m.npair;p++) m.pair[p].fofs = m.pair[p].sofs; m.nfw = 1; }
  else { int fo = 0; for(int p=0;p<m.npair;p++){ m.pair[p].fofs = fo; fo += (m.cell[m.pair[p].cell].nvert + 31) & ~31; } m.nfw = fo/32; }
  if( m.nfw > MAX_FWORDS ){ err = "too many contact flag words (MAX_FWORDS)"; return false; }
  if( m.nfw < 1 ) m.nfw = 1;
  /* links that take an external wrench (rkFDBatchSetExtWrenchLinks): row k of the input is link fext_links[k].  The wrench
   * comes in world axes, so such a world propagates the world frames */
  if( (int)w.fext_links.size() > MAX_LINKS ){ err = "at most " + std::to_string(MAX_LINKS) + " links take an external wrench (MAX_LINKS)"; return false; }
  for(size_t k=0;k<w.fext_links.size();k++){
    const int i = w.fext_links[k];
    if( i < 0 || i >= nl ){ err = "external wrench: link index " + std::to_string(i) + " out of range [0, " + std::to_string(nl) + ")"; return false; }
    if( m.link[i].fext_row >= 0 ){ err = "external wrench: link " + std::to_string(i) + " listed twice"; return false; }
    m.link[i].fext_row = (int)k;
  }
  m.nfext = (int)w.fext_links.size();
  m.need_world = m.npair > 0 || m.nfext > 0;

  /* ---- topology flags and the scratch slot map */
  for(int i=0;i<nl;i++) if( m.link[i].parent >= 0 ) m.link[m.link[i].parent].nchild++;
  for(int i=0;i<nl;i++){ LinkDev &d = m.link[i]; d.serial = ( d.parent >= 0 && d.parent == i-1 && m.link[d.parent].nchild == 1 ) ? 1 : 0;
    d.branch_slot = d.accum_slot = d.wext_slot = d.frame_slot = -1; }
  model_layout(m, false);
  /* ---- rigid-contact tables: slot -> (pair, vertex), workspace layout per warp */
  m.rigid_mask = 0; int nrs = 0;
  if( m.has_rigid && m.solver != S_VOLUME && m.nslot > RIGID_MAX_SLOTS ){
    err = "the rigid vertex solvers (MLCP, Vert) handle at most 32 contact slots per environment (cell vertices x boxes of static links and, for rigid contact info, of other moving links)"; return false; }
  for(int p=0;p<m.npair;p++) for(int k=0;k<m.cell[m.pair[p].cell].nvert;k++){
    const int sidx = m.pair[p].sofs + k;
    if( sidx < RIGID_MAX_SLOTS ){ m.slot_pair[sidx] = p; m.slot_vert[sidx] = k; }
    if( m.pair[p].type == C_RIGID ){ if( sidx < 32 ) m.rigid_mask |= 1ull << (2*sidx); nrs++; }
  }
  m.nmax = 3*nrs; m.ws_doubles = 0;
  /* single-link MLCP path (Core::rigid_mlcp_single): every rigid slot on one link */
  m.rigid_link = -1; m.ws1_doubles = 0;
  m.nrg = 0;
  if( m.has_rigid ){
    /* contact groups: links with rigid cells, at most MAX_RG of them, pairwise in different chains */
    int lk = -2; bool ok = true;
    for(int p=0;p<m.npair && ok;p++) if( m.pair[p].type == C_RIGID ){
      const int l = m.cell[m.pair[p].cell].link; bool seen = false;
      for(int g=0;g<m.nrg;g++) if( m.rg_link[g] == l ) seen = true;
      if( seen ) continue;
      if( m.nrg >= MAX_RG ){ ok = false; break; }
      int root = l; while( m.link[root].parent >= 0 ) root = m.link[root].parent;
      for(int g=0;g<m.nrg;g++){ int r2 = m.rg_link[g]; while( m.link[r2].parent >= 0 ) r2 = m.link[r2].parent; if( r2 == root ) ok = false; }
      m.rg_link[m.nrg++] = l;
    }
    if( m.rigid_moving ) ok = false;             /* a rigid pair of two moving links: the dense path (A couples them) */
    lk = ( ok && m.nrg > 0 ) ? m.rg_link[0] : -1;
    if( !ok ) m.nrg = 0;
    bool lpos = true;           /* the Vert path divides by the relaxation of every rigid pair */
    for(int p=0;p<m.npair;p++) if( m.pair[p].type == C_RIGID && !(m.pair[p].L > 0.0) ) lpos = false;
    if( lk >= 0 && m.solver == S_MLCP ){ m.rigid_link = lk; m.ws1_doubles = W1_CT + W1_CTN*nrs; }
    if( lk >= 0 && m.solver == S_VERT && lpos && m.pyramid <= 12 ){ m.rigid_link = lk; m.ws1_doubles = W1_CT + W1_CTN*nrs + QP_HIST*qp_hist_stride(nrs); }
    if( m.rigid_link < 0 ) m.nrg = 0;
  }
  if( m.has_rigid && m.solver == S_VOLUME ){
    /* the Volume solver (rkfd_volume.cuh) works on thread-local data: no workspace.  Contact volumes are formed for cells
     * with the 8 corners of a box (parallelepiped; the soles of mighty.ztk); other rigid cells are watched only - an
     * environment in which one of them touches is flagged (status bit 8).  At least one box cell must exist. */
    int nvb = 0;
    for(int p=0;p<m.npair;p++) if( m.pair[p].type == C_RIGID ){
      const CellDev &c = m.cell[m.pair[p].cell];
      m.pair[p].volbox = ( c.nvert == 8 && box_sign_bit_order(m.vert + 3*c.vofs) ) ? 1 : 0; nvb += m.pair[p].volbox;
    }
    if( nvb == 0 ){ err = "Volume solver: no rigid cell has the 8 corners of a box (parallelepiped) - contact volumes are formed for box cells only"; return false; }
    m.ws_doubles = 0; m.ws_geo = m.ws_b = m.ws_f = m.ws_A = m.ws_du = m.ws_da = m.ws_qp = 0;
    return true;
  }
  if( m.has_rigid ){
    const int n = m.nmax, mc = m.pyramid*nrs, nm = n + mc; int o = 0;
    m.ws_geo = o; o += GEO_DOUBLES*nrs;
    m.ws_b = o;  o += n;
    m.ws_f = o;  o += n;
    m.ws_A = o;  o += n*n;
    m.ws_du = o; o += n*6*nl;         /* per probe column: joint-space increments, 6 per link (Core::probe indexes du0 + 6*link: with n*nl
                                       * the columns >= n/6 overlapped the acceleration increments of other columns and were correct only
                                       * in lockstep) */
    m.ws_da = o; o += n*6*nl;         /* per probe column: link acceleration increments */
    m.ws_qp = o;
    (void)nm;
    if( m.solver == S_VERT ) o += 2*n*n + 4*n + 3*mc + mc + n*mc + 2*mc*mc + 3*mc + 32*(mc+1) + (mc+2) + 64;   /* layout in Core::qp_vert */
    m.ws_doubles = (o + 31) & ~31;
  }
  return true;
}

bool kin_table(const ModelDev &m, int nlink, const int *links, KinDev &t, std::string &err)
{
  std::memset(&t, 0, sizeof t);
  if( nlink < 0 ){ err = "the number of links must be >= 0"; return false; }
  if( nlink > MAX_LINKS ){ err = "at most " + std::to_string(MAX_LINKS) + " links per call (MAX_LINKS)"; return false; }
  if( !links && nlink != m.nl ){ err = "links == NULL (all links) needs nlink == " + std::to_string(m.nl); return false; }
  for(int k=0;k<nlink;k++){ const int i = links ? links[k] : k;
    if( i < 0 || i >= m.nl ){ err = "link index " + std::to_string(i) + " out of range [0, " + std::to_string(m.nl) + ")"; return false; } }
  /* links to visit: the requested ones and their ancestors (parents precede children in the model) */
  bool need[MAX_LINKS] = {false};
  for(int k=0;k<nlink;k++) for(int i = links ? links[k] : k; i >= 0 && !need[i]; i = m.link[i].parent) need[i] = true;
  int pos[MAX_LINKS];
  for(int i=0;i<m.nl;i++){
    const LinkDev &d = m.link[i]; KinLinkDev &l = t.link[i];
    std::memcpy(l.Ro, d.Ro, sizeof l.Ro); std::memcpy(l.po, d.po, sizeof l.po);
    l.cls = d.rcls; l.sg = d.rcls == RO_RXP ? 1.0 : ( d.rcls == RO_RXM ? -1.0 : 0.0 ); l.pz = d.pz;
    l.parent = d.parent; l.jtype = d.jtype; l.qofs = d.qofs; l.keep = -1; l.omask = 0u;
    if( d.jtype == J_BRFLOAT ) t.brk = 1;
    pos[i] = -1;
    if( need[i] ){ pos[i] = t.nwalk; t.walk[t.nwalk++] = i; }
  }
  for(int k=0;k<nlink;k++) t.link[links ? links[k] : k].omask |= 1u << k;
  t.nsel = nlink;
  /* a parent that is not the link visited just before its child is read back from a keep slot; slots are reused once their
   * last reader has loaded them */
  int last[MAX_LINKS];
  for(int i=0;i<MAX_LINKS;i++) last[i] = -1;
  for(int w=0; w<t.nwalk; w++){ const int i = t.walk[w], p = m.link[i].parent;
    if( p >= 0 && ( w == 0 || t.walk[w-1] != p ) ) last[p] = w; }
  int owner[MAX_LINKS];      /* slot -> link kept there, -1 free */
  for(int s=0;s<MAX_LINKS;s++) owner[s] = -1;
  for(int w=0; w<t.nwalk; w++){
    for(int s=0;s<t.nkeep;s++) if( owner[s] >= 0 && last[owner[s]] <= w ) owner[s] = -1;
    const int i = t.walk[w];
    if( last[i] < 0 ) continue;
    int s = 0; while( owner[s] >= 0 ) s++;
    owner[s] = i; t.link[i].keep = s; if( s + 1 > t.nkeep ) t.nkeep = s + 1;
  }
  return true;
}

}  // namespace rkfd
