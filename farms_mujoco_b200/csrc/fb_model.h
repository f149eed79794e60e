/*
 * fb_model.h -- device-side model tables of the batched FARMS stepping engine.
 *
 * FbModel/FbFarms (include/farms_b200.h, float64 host arrays) are flattened by
 * fb_build_model() into two blobs (int32 + float32) plus a table of offsets;
 * the same DevModel struct is handed to the CUDA kernels by value and to the
 * host emulation build used by the CPU unit tests (tests/emu).  Plain C++,
 * no CUDA headers.
 *
 * What the tables describe follows the MuJoCo subset of SURVEY.md Appendix A
 * (reference call sites: farms_mujoco/simulation/simulation.py:53,156) and the
 * farms index maps of farms_mujoco/simulation/physics.py:188-393.
 */
#ifndef FB_MODEL_H_
#define FB_MODEL_H_

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/farms_b200.h"

/* MuJoCo constants (third party; isolated here, mirrored in mjcf_subset.py) */
#define FB_MINVAL 1e-15f
#define FB_MINIMP 0.0001f
#define FB_MAXIMP 0.9999f

/* offsets (in elements) into the int blob I and the float blob F */
struct DevOffsets {
  /* ints */
  int body_parent, body_jnt, body_dofadr, body_dofnum, body_firstchild, body_nextsib,
      body_lastdof, body_ancmask, lvl_start, lvl_body, body_anc, body_size;
  int jnt_type, jnt_body, jnt_qposadr, jnt_dofadr, jnt_limited, jnt_actstart, act_sorted;
  int dof_body, dof_jnt, dof_parent, dof_Madr, dof_nanc;
  int ent_i, ent_j;
  int col_start, col_ent, col_dof;   /* per dof: entries (e, d) of descendants d whose row holds it */
  int st_pivstart, st_piv, fop_start, fop, sop_start, sop;   /* elimination schedule */
  int cand_body, cand_iscapsule, cand_sensor;
  int cand_body1;  /* int [ncand] the body of geom1: 0 (the world) for plane candidates, the first sphere's body for pair candidates (kind 9) */
  int act_jnt, act_ctrllimited, act_forcelimited;
  int link_body, fj_qposadr, fj_dofadr, fj_jntid, fj_actpos, fj_actvel, fj_acttrq, xfrc_body,
      swim_link, swim_xfrc, body_xfrcrow, wc_act;
  /* floats */
  int body_pos, body_quat, body_ipos, body_iquat, body_mass, body_inertia, body_invw;
  int jnt_pos, jnt_axis, jnt_stiffness, jnt_range, jnt_margin, jnt_solref, jnt_solimp, jnt_qpos0;
  int dof_damping, dof_armature, dof_invw;
  int cand_gquat;  /* float [ncand][4] geom orientation in the body frame (ellipsoids; identity otherwise) */
  int cand_lpos, cand_laxis, cand_radius, cand_pn, cand_pd, cand_friction, cand_solref,
      cand_solimp, cand_margin, cand_gap, cand_invw;
  int act_gain, act_bias, act_ctrlrange, act_forcerange, act_gear;
  int swim_mass, swim_height, swim_density, swim_coef;
  int wc_amp, wc_freq, wc_lag, wc_off;
  int key_qpos, key_qvel;
  /* tables of the environment-per-thread path (fb_fast.h) */
  int ft_actwc;   /* int   [nu] wave index of an actuator, -1 */
  int ft_actoff;  /* int   [nu] 1: force-limited to [0, 0] (contributes nothing) */
  int ft_chk;     /* float [nchk][4] conservative plane checks (normal, offset) */
  /* tables of the per-thread constrained step (fb_fastc.h) */
  int ft_sstart;  /* int   [n_contacts+1] contact sensor -> entries (CandRec index, sign) it sums (sensors.pyx:140-190) */
  int ft_scand;   /* int   [...] */
  int ft_ssign;   /* float [...] */
};

/* ---- environment-per-thread path (fb_fast.h) ------------------------------------ */
#define FB_FAST_MAXBODY 64
/* flags of FastRec */
#define FT_ADD_CARRY 1      /* child b+1 hands its articulated inertia over in registers */
#define FT_HAS_SLOT 2       /* has children that are not b+1: they accumulate into slot `slot` */
#define FT_TO_CARRY 4       /* parent is b-1 */
#define FT_FIRST_WRITER 8   /* first child (descending order) to write the parent's slot */
#define FT_LIMITED 16
#define FT_ACT_SIMPLE 32    /* unclamped actuators, gear 1, all logged: one linear form */
#define FT_HAS_WAVE 64
#define FT_HAS_JPOS 128
/* bits 24..30: 1 + row of the joint's spring reference behind the nu ctrl rows of a control-sequence
 * step (fb_set_cpg_springrefs); 0: the joint's spring reference is qpos_spring */
#define FT_SREF_SHIFT 24
#define FT_SREF(flags_) ((((flags_) >> FT_SREF_SHIFT) & 0x7f) - 1)
#define FB_MAX_SPRINGREFS 126
#define FT_AXISYM 256        /* inertia = Ib[0]*1 + Ib[1]*n n', n = Ib[2..4] (capsule, cylinder, sphere) */

/* Everything the recursion needs about one body, resolved at model build: no index
 * chasing in the kernel.  The table travels in the kernel parameters (constant bank),
 * so every lane of a warp reads it with uniform, hoistable loads.  72 words = nine 32-byte lines:
 * keep it that size (a 73rd word cost the swimming kernel 3 %, r3a). */
struct FastRec {
  int32_t parent, jtype, qa, da;          /* joint type -1: welded; qa/da: qpos/qvel address */
  int32_t flags, slot, pslot, link;       /* link: farms link row, -1 */
  int32_t fj, xr, swim, jid;              /* farms joint row, xfrc row, swim index, joint id */
  int32_t chk0, chk1, wave_act, pblk;     /* plane-check range; ctrl index the wave writes; FB_NF*(parent-1) */
  float dpos[3], mass;                    /* body_pos - jnt_pos(parent); body mass */
  float bquat[4];
  float axis[3], qpos0;
  float jpos[3], margin;
  float lo, hi, stiffness, damping;
  float armature, Kq, Kqd, T0;            /* simple actuation: T0 + Kq q + Kqd qd (+ ctrl terms) */
  float hloc[3], wgain;                   /* com - anchor (body axes); gear*gain of the wave actuator */
  float Ib[6], wfreq, wlag;               /* inertia about the com, body axes (xx yy zz xy xz yz) */
  float wamp, woff, lift, height;         /* lift = 1000*9.81*mass/density (drag.pyx:142-145) */
  float coef[6], KqU, KqdU;               /* KqU/KqdU/T0U: the part of the actuation that the */
  float T0U;                              /* farms joint_torque column does not log */
  int32_t bc0, bc1, pblk7;                /* candidates of the body: CandRec[bc0 .. bc1) (fb_fastc.h); 7*(parent-1) (SLIM blocks) */
  float chk[4];                           /* first conservative plane check (normal, offset) */
};

/* Tree split of the unconstrained kernel for SMALL batches (fb_fast.h, FbFast<.., SPLIT = 1>): the 32
 * environments of a warp are stepped by `nwarps` warps that share their shared-memory blocks, each
 * visiting its own bodies -- the trunk up to the last branching body on warp 0 (phase A), then,
 * after a block barrier, the subtrees hanging off it in parallel (phase B: the rest of the trunk
 * stays on warp 0, subtrees with the same parent share a warp).  Leaves -> root sweeps run the lists
 * backwards, phase B first.  A launch is then about one trunk + one subtree long instead of the whole
 * tree.  order[w][0 .. n[w]) ascending, phase A = [0, boundary[w]). */
#define FB_SPLIT_MAXW 4
struct FastSplit {
  int32_t nwarps, n[FB_SPLIT_MAXW], boundary[FB_SPLIT_MAXW];
  uint8_t order[FB_SPLIT_MAXW][FB_FAST_MAXBODY];
};

/* One collision candidate (world plane vs sphere / capsule end) of the per-thread constrained
 * step (fb_fastc.h), in body order; travels in the kernel parameters like FastRec.  16 words. */
#define FB_FAST_MAXCAND 112
struct CandRec {
  int32_t body, cid, iscapsule, pblk;     /* cid: index into the cand_* tables; pblk = FB_NF*(body-1);
                                           * iscapsule: 0 sphere, 1 capsule end, 2 box corner, 3 first corner of a box,
                                           * 4 ellipsoid (laxis = radii; radius, pad[0], pad[1] = x, y, z of the
                                           * geom's orientation quaternion in the body frame, w >= 0),
                                           * 5..8 cylinder points (laxis = x, y, z of that quaternion; radius,
                                           * pad[0] = half length) */
  float pn[3], mu;                        /* plane normal (world), friction */
  float lpos[3], radius;                  /* centre relative to the body's joint anchor (body axes) */
  float laxis[3], pd;                     /* capsule axis (body axes) / box centre relative to the anchor; plane offset */
  float includemargin, invw, pad[2];
};

/* per-environment shared-memory layout, in floats; element i of an environment lives at
 * i*BLOCK + thread.  One block of FB_NF floats per moving body (pose and velocity), then
 * the accumulation slots; the floating root's qpos/qvel live in registers. */
enum { FB_QUAT = 0, FB_ORG = 4, FB_VEL = 7, FB_NF = 13 };
/* second half of the per-body state, kept in an L2-resident global scratch (element i of
 * thread t at i*n_threads + t: coalesced) so that four warps of environments fit one SM */
enum { FG_W = 0, FG_U = 6, FG_DINV = 7, FG_TRQ = 8, FG_Q = 9, FG_QD = 10, FG_TC = 11, FG_TU = 12,
       FG_NF = 13 };
struct DevFastLayout {
  int ok;          /* 1 when the model fits the path's subset */
  int body0, slots;
  int nslot, n_float;   /* shared floats per environment */
  int n_scratch;        /* global scratch floats per environment */
  int jrow_std;         /* farms joint row = 18 columns, position 0, velocity 1, torque 11 */
  int coop_io;          /* [32][nq + nv + nu + 6 nbody] fits the warp's shared memory: tiled state I/O */
  int coop_io2;         /* SLIM layout: [32][nq + nv + nu] and [32][6 nbody] each fit: two-phase tiled state I/O */
  int n_float_slim, n_scratch_slim;   /* SLIM variant of the unconstrained kernel (fb_fast.h) */
  int n_con;            /* global scratch floats per environment of the constrained step (fb_fastc.h) */
  int con_ok;           /* 1 when the per-thread constrained step covers the model (else: team kernel) */
  int lean;             /* 1: hinge joints only, anchors at the body origins, axisymmetric inertias, the linear
                         * actuation form on every joint, farms joints-row layout (FbFast<.., LEAN = 1>) */
};

/* scratch of the per-thread constrained step (fb_fastc.h), element i of thread t at i*BLK + t:
 * one block per moving body, one for the floating root, one per collision candidate */
enum { NB_U = 0, NB_DINV = 6, NB_UU = 7, NB_AP = 8, NB_A = 14, NB_MD = 15, NB_P = 16, NB_MP = 17,
       NB_DLO = 18, NB_DHI = 19, NB_ARLO = 20, NB_ARHI = 21, NB_LIMF = 22, NB_TAUC = 23, NB_NF = 24 };
enum { NR_A = 0, NR_MD = 6, NR_P = 12, NR_MP = 18, NR_NF = 24 };
enum { NC_R = 0, NC_T1 = 3, NC_D = 6, NC_RES = 7, NC_JP = 10, NC_POS = 13, NC_NF = 16 };

/* per-environment shared-memory layout (float offsets; component-major SoA:
 * element (k, i) of an array with N items lives at off + k*N + i) */
struct DevLayout {
  int qpos, qvel, ctrl, actf, xpos, xquat, xipos, xanchor, xaxis, cinert, cdof, cvel, xfrc,
      qM, qLD, dinv, fsm, qacc, fcon, grad, pvec, tmp1, tmp2, limf, scratch;
  /* aliases inside scratch */
  int crb, cacc, cfrc, buf, altB, Md, H;
  /* hard normal rows of frictionless pairs (n_hard of them): V = H^-1 Jn' [n_hard][nv], S = Jn V and
   * its Cholesky factor [n_hard][n_hard] each, multipliers, residuals Jn a - aref, their tolerances
   * and the right-hand side of S lambda = Jn u - x [n_hard] each */
  int hV, hS, hL, hlam, hx, htol, hrhs;
  int n_float;   /* floats per env */
  int con_cand;  /* int region: con_cand[maxcon] */
  int hcon, hon, hws;   /* int regions [n_hard]: contact of each active hard row, working-set flags, compact working set */
  int n_int;
};

struct DevModel {
  int nbody, njnt, nq, nv, nu, ncand, nM, nlevel, nmaskw;
  int nstage, sched_team;
  int nround_anc, nround_sub; /* pointer-jumping rounds (ancestors), doubling rounds (subtrees) */    /* stages of the scheduled sparse factor/solve; lanes it was built for */
  int n_links, n_joints, n_contacts, n_xfrc, n_swim, n_wc;
  int maxcon, maxefc, npack; /* npack = nv*(nv+1)/2 */
  int n_pair;                /* candidates of explicit <pair>s (two-body rows: team kernel only, dense Newton Hessian) */
  int n_hard;                /* ... of them frictionless, solved as hard normal rows (kind 10; H stays tree-sparse) */
  int solver_iterations, any_damping, any_stiffness, any_limit;
  int col_jpos, col_jvel, col_jtrq, col_jlim;
  int link_cols, joint_cols, contact_cols, xfrc_cols;
  int water_drag, water_buoyancy;
  float timestep, grav[3], impratio, inv_total_mass, solver_scale, tolerance;
  float water_surface, water_viscosity, water_velocity[3];
  /* log scaling: value_SI = value_sim * inv_<unit> (physics.py:428-523) */
  float inv_meters, inv_velocity, inv_angvel, inv_torques, inv_newtons;
  float newtons, torques;
  const int32_t *I;
  const float *F;
  DevOffsets o;
  DevLayout L;
  DevFastLayout X;
};

/* ---------------------------------------------------------------- builder */
struct FbHostModel {
  std::vector<int32_t> I;
  std::vector<float> F;
  DevModel m;  /* I/F pointers left null; the caller patches them */
  std::vector<FastRec> rec;   /* [nbody] when m.X.ok */
  std::vector<CandRec> crec;  /* [ncand] in body order when m.X.con_ok */
  FastSplit split;            /* nwarps = 1: the tree does not branch (or the model is outside the path) */
  std::string error;
};

/* Phase schedule of FastSplit for a tree given by parent[] (parent[b] < b, body 0 = world). */
inline void fb_build_split(const std::vector<int> &parent, int max_warps, FastSplit &sp) {
  const int nb = (int)parent.size();
  std::memset(&sp, 0, sizeof(sp));
  sp.nwarps = 1;
  for (int b = 1; b < nb; b++) sp.order[0][sp.n[0]++] = (uint8_t)b;
  sp.boundary[0] = sp.n[0];
  if (nb < 4 || nb > FB_FAST_MAXBODY || max_warps < 2) return;
  /* the last body some other body branches off (a child that is not its successor) */
  int split = 0;
  for (int b = 2; b < nb; b++)
    if (parent[b] >= 1 && parent[b] != b - 1 && parent[b] > split) split = parent[b];
  if (split < 1 || split >= nb - 1) return;
  /* phase B: the forest on the bodies after `split`; a component is named by its first body, and
   * components whose roots share a parent are merged (their hand-overs accumulate in one slot) */
  std::vector<int> comp(nb, -1);
  std::vector<std::vector<int>> groups;
  std::vector<int> group_parent;
  for (int b = split + 1; b < nb; b++) {
    const int p = parent[b];
    if (p > split) { comp[b] = comp[p]; groups[comp[b]].push_back(b); continue; }
    int g = -1;
    /* the successor of `split` continues warp 0's chain in registers: a group of its own */
    if (!(b == split + 1 && p == split))
      for (size_t k = 0; k < groups.size(); k++) if (group_parent[k] == p) g = (int)k;
    if (g < 0) { g = (int)groups.size(); groups.emplace_back(); group_parent.push_back(b == split + 1 && p == split ? -1 : p); }
    comp[b] = g;
    groups[g].push_back(b);
  }
  if (groups.size() < 2) return;
  const int nw = (int)groups.size() < max_warps ? (int)groups.size() : max_warps;
  std::vector<std::vector<int>> phase_b(nw);
  std::vector<int> load(nw, 0);
  std::vector<char> done(groups.size(), 0);
  for (size_t k = 0; k < groups.size(); k++)
    if (group_parent[k] == -1) { phase_b[0] = groups[k]; load[0] = (int)groups[k].size(); done[k] = 1; }
  for (;;) {                                   /* largest remaining group to the least loaded warp */
    int best = -1;
    for (size_t k = 0; k < groups.size(); k++)
      if (!done[k] && (best < 0 || groups[k].size() > groups[best].size())) best = (int)k;
    if (best < 0) break;
    int w = 0;
    for (int k = 1; k < nw; k++) if (load[k] < load[w]) w = k;
    phase_b[w].insert(phase_b[w].end(), groups[best].begin(), groups[best].end());
    load[w] += (int)groups[best].size();
    done[best] = 1;
  }
  std::memset(&sp, 0, sizeof(sp));
  sp.nwarps = nw;
  for (int b = 1; b <= split; b++) sp.order[0][sp.n[0]++] = (uint8_t)b;
  sp.boundary[0] = sp.n[0];
  for (int w = 0; w < nw; w++) {
    std::sort(phase_b[w].begin(), phase_b[w].end());
    for (int b : phase_b[w]) sp.order[w][sp.n[w]++] = (uint8_t)b;
  }
}

namespace fbdetail {
inline int put_i(std::vector<int32_t> &I, const std::vector<int32_t> &v) {
  int off = (int)I.size();
  I.insert(I.end(), v.begin(), v.end());
  if (v.empty()) I.push_back(0);
  return off;
}
inline int put_f(std::vector<float> &F, const std::vector<double> &v) {
  int off = (int)F.size();
  for (double x : v) F.push_back((float)x);
  if (v.empty()) F.push_back(0.f);
  while (F.size() % 4) F.push_back(0.f);
  return off;
}
inline std::vector<int32_t> vi(const int32_t *p, int n) { return std::vector<int32_t>(p, p + n); }
inline std::vector<double> vd(const double *p, int n) { return std::vector<double>(p, p + n); }
inline void quat2mat(const double *q, double *m) {
  double w = q[0], x = q[1], y = q[2], z = q[3];
  m[0] = w*w + x*x - y*y - z*z; m[1] = 2*(x*y - w*z);         m[2] = 2*(x*z + w*y);
  m[3] = 2*(x*y + w*z);         m[4] = w*w - x*x + y*y - z*z; m[5] = 2*(y*z - w*x);
  m[6] = 2*(x*z - w*y);         m[7] = 2*(y*z + w*x);         m[8] = w*w - x*x - y*y + z*z;
}
}  // namespace fbdetail

/* Flatten FbModel + FbFarms.  Returns false and sets out.error when the model
 * leaves the supported subset. */
inline bool fb_build_model(const FbModel *fm, const FbFarms *ff, const FbWaveController *wc,
                           int team, FbHostModel &out) {
  using namespace fbdetail;
  DevModel &m = out.m;
  std::memset(&m, 0, sizeof(m));
  std::vector<int32_t> &I = out.I;
  std::vector<float> &F = out.F;
  I.clear(); F.clear();
  const int nb = fm->nbody, nj = fm->njnt, nv = fm->nv, nu = fm->nu, nc = fm->ncand;
  if (nb < 2 || nv < 1) { out.error = "model has no moving body"; return false; }
  m.nbody = nb; m.njnt = nj; m.nq = fm->nq; m.nv = nv; m.nu = nu; m.ncand = nc; m.nM = fm->nM;
  m.timestep = (float)fm->timestep;
  for (int k = 0; k < 3; k++) m.grav[k] = (float)fm->gravity[k];
  m.impratio = (float)fm->impratio;
  m.solver_iterations = fm->solver_iterations > 0 ? fm->solver_iterations : 100;
  m.tolerance = (float)fm->tolerance;
  m.solver_scale = (float)(1.0/(fm->meaninertia*(nv > 1 ? nv : 1)));

  /* tree tables */
  std::vector<int32_t> depth(nb, 0), firstchild(nb, -1), nextsib(nb, -1), lastchild(nb, -1),
      lastdof(nb, -1);
  int roots = 0, maxdepth = 0;
  double total_mass = 0;
  for (int b = 1; b < nb; b++) {
    int p = fm->body_parentid[b];
    if (p < 0 || p >= b) { out.error = "bodies must be in depth-first order"; return false; }
    if (p == 0) roots++;
    depth[b] = depth[p] + 1;
    if (depth[b] > maxdepth) maxdepth = depth[b];
    if (lastchild[p] < 0) firstchild[p] = b; else nextsib[lastchild[p]] = b;
    lastchild[p] = b;
    lastdof[b] = fm->body_dofnum[b] > 0 ? fm->body_dofadr[b] + fm->body_dofnum[b] - 1 : lastdof[p];
    total_mass += fm->body_mass[b];
  }
  if (roots != 1) { out.error = "exactly one kinematic tree is supported (static bodies must be fused)"; return false; }
  m.inv_total_mass = total_mass > 1e-15 ? (float)(1.0/total_mass) : 0.f;
  m.nlevel = maxdepth;
  std::vector<int32_t> lvl_start(maxdepth + 1, 0), lvl_body;
  for (int l = 1; l <= maxdepth; l++) {
    lvl_start[l-1] = (int)lvl_body.size();
    for (int b = 1; b < nb; b++) if (depth[b] == l) lvl_body.push_back(b);
  }
  lvl_start[maxdepth] = (int)lvl_body.size();
  m.nmaskw = (nv + 31)/32;
  std::vector<int32_t> ancmask((size_t)nb*m.nmaskw, 0);
  for (int b = 1; b < nb; b++)
    for (int d = lastdof[b]; d >= 0; d = fm->dof_parentid[d])
      ancmask[(size_t)b*m.nmaskw + d/32] |= (int32_t)(1u << (d % 32));

  DevOffsets &o = m.o;
  o.body_parent = put_i(I, vi(fm->body_parentid, nb));
  o.body_jnt = put_i(I, vi(fm->body_jntid, nb));
  o.body_dofadr = put_i(I, vi(fm->body_dofadr, nb));
  o.body_dofnum = put_i(I, vi(fm->body_dofnum, nb));
  o.body_firstchild = put_i(I, firstchild);
  o.body_nextsib = put_i(I, nextsib);
  o.body_lastdof = put_i(I, lastdof);
  o.body_ancmask = put_i(I, ancmask);
  o.lvl_start = put_i(I, lvl_start);
  o.lvl_body = put_i(I, lvl_body);
  /* pointer jumping: body_anc[r*nb + b] = 2^r-th ancestor of b (world absorbs) */
  {
    int R = 0;
    while ((1 << R) < maxdepth) R++;
    m.nround_anc = R;
    std::vector<int32_t> anc((size_t)(R > 0 ? R : 1)*nb, 0);
    for (int b = 0; b < nb; b++) anc[b] = b > 0 ? fm->body_parentid[b] : 0;
    for (int r = 1; r < R; r++)
      for (int b = 0; b < nb; b++) anc[(size_t)r*nb + b] = anc[(size_t)(r-1)*nb + anc[(size_t)(r-1)*nb + b]];
    o.body_anc = put_i(I, anc);
    /* subtree sizes; subtrees must be contiguous id ranges (depth-first preorder) */
    std::vector<int32_t> size(nb, 1);
    for (int b = nb - 1; b > 0; b--) size[fm->body_parentid[b]] += size[b];
    int maxsize = 1;
    for (int b = 1; b < nb; b++) {
      for (int c = b + 1; c < b + size[b]; c++) {
        int a = c;
        while (a > b) a = fm->body_parentid[a];
        if (a != b) { out.error = "bodies are not in depth-first preorder"; return false; }
      }
      if (size[b] > maxsize) maxsize = size[b];
    }
    int R2 = 0;
    while ((1 << R2) < maxsize) R2++;
    if ((1 << R2) == maxsize) R2++;     /* bit R2-1 must be able to hold maxsize */
    m.nround_sub = R2;
    o.body_size = put_i(I, size);
  }

  /* joints + actuators grouped by joint */
  std::vector<int32_t> actstart(nj + 1, 0), act_sorted;
  for (int j = 0; j < nj; j++) {
    actstart[j] = (int)act_sorted.size();
    for (int a = 0; a < nu; a++) if (fm->actuator_trnid[a] == j) act_sorted.push_back(a);
  }
  actstart[nj] = (int)act_sorted.size();
  std::vector<double> jqpos0(nj, 0.0);
  m.any_limit = 0; m.any_stiffness = 0;
  for (int j = 0; j < nj; j++) {
    jqpos0[j] = fm->qpos0[fm->jnt_qposadr[j]];
    if (fm->jnt_type[j] == FB_JNT_BALL) { out.error = "ball joints are outside the FARMS schema"; return false; }
    if (fm->jnt_limited[j] && fm->jnt_type[j] != FB_JNT_FREE) m.any_limit = 1;
    if (fm->jnt_stiffness[j] != 0) m.any_stiffness = 1;
  }
  o.jnt_type = put_i(I, vi(fm->jnt_type, nj));
  o.jnt_body = put_i(I, vi(fm->jnt_bodyid, nj));
  o.jnt_qposadr = put_i(I, vi(fm->jnt_qposadr, nj));
  o.jnt_dofadr = put_i(I, vi(fm->jnt_dofadr, nj));
  o.jnt_limited = put_i(I, vi(fm->jnt_limited, nj));
  o.jnt_actstart = put_i(I, actstart);
  o.act_sorted = put_i(I, act_sorted);

  /* dofs + sparse mass-matrix entry table */
  std::vector<int32_t> nanc(nv, 0), ent_i(fm->nM, 0), ent_j(fm->nM, 0);
  m.any_damping = 0;
  for (int d = 0; d < nv; d++) {
    int adr = fm->dof_Madr[d];
    for (int a = d; a >= 0; a = fm->dof_parentid[a]) {
      if (adr >= fm->nM) { out.error = "dof_Madr/nM mismatch"; return false; }
      ent_i[adr] = d; ent_j[adr] = a; adr++; nanc[d]++;
    }
    if (fm->dof_damping[d] > 0) m.any_damping = 1;
  }
  o.dof_body = put_i(I, vi(fm->dof_bodyid, nv));
  o.dof_jnt = put_i(I, vi(fm->dof_jntid, nv));
  o.dof_parent = put_i(I, vi(fm->dof_parentid, nv));
  o.dof_Madr = put_i(I, vi(fm->dof_Madr, nv));
  o.dof_nanc = put_i(I, nanc);
  o.ent_i = put_i(I, ent_i);
  o.ent_j = put_i(I, ent_j);
  {
    /* column view of the tree-sparse matrix: M x needs, for dof j, the entries M[d][j] of its
     * descendants d (the row view gives the ancestors) */
    std::vector<int32_t> cstart(nv + 1, 0), cent, cdof_;
    for (int j = 0; j < nv; j++) {
      cstart[j] = (int)cent.size();
      for (int e = 0; e < fm->nM; e++)
        if (ent_j[e] == j && ent_i[e] != j) { cent.push_back(e); cdof_.push_back(ent_i[e]); }
    }
    cstart[nv] = (int)cent.size();
    o.col_start = put_i(I, cstart);
    o.col_ent = put_i(I, cent);
    o.col_dof = put_i(I, cdof_);
  }

  /* Scheduled sparse L'DL and back-substitution.  Pivots are grouped into stages by
   * tree depth (deepest first): every pivot of a stage has all its descendants
   * eliminated, pivots of one stage lie in different branches.  Within a stage the
   * update operations are grouped by destination and each group is pinned to one lane,
   * so concurrent lanes never write the same word and the summation order is fixed
   * (bit-reproducible).  Factor op: qLD[dst] -= qLD[a]*qLD[b]*dinv[piv];
   * solve op: x[dst] -= qLD[adr]*y[piv]. */
  {
    if (team < 1) team = 1;
    int maxdd = 0;
    for (int d = 0; d < nv; d++) if (nanc[d] > maxdd) maxdd = nanc[d];
    const int NS = maxdd;
    m.nstage = NS; m.sched_team = team;
    std::vector<int32_t> pivstart(NS + 1, 0), piv;
    std::vector<int32_t> fstart((size_t)NS*team + 1, 0), fops, sstart((size_t)NS*team + 1, 0), sops;
    for (int st = 0; st < NS; st++) {
      int depth = maxdd - st;
      pivstart[st] = (int)piv.size();
      struct Op { int dst, a, b, k; };
      std::vector<Op> f, sv;
      for (int k = 0; k < nv; k++) {
        if (nanc[k] != depth) continue;
        piv.push_back(k);
        int adr = fm->dof_Madr[k], nk = nanc[k];
        for (int s1 = 1; s1 < nk; s1++) {
          int as = ent_j[adr + s1], ra = fm->dof_Madr[as];
          for (int t = s1; t < nk; t++) f.push_back({ra + t - s1, adr + s1, adr + t, k});
          sv.push_back({as, adr + s1, 0, k});
        }
      }
      auto distribute = [&](std::vector<Op> &ops, std::vector<int32_t> &start,
                            std::vector<int32_t> &words) {
        /* group by dst, largest groups first, each to the currently lightest lane */
        std::vector<std::vector<Op>> groups;
        std::vector<int> where(65536, -1);
        for (const Op &op : ops) {
          if (where[op.dst] < 0) { where[op.dst] = (int)groups.size(); groups.emplace_back(); }
          groups[where[op.dst]].push_back(op);
        }
        std::vector<int> order(groups.size());
        for (size_t i = 0; i < order.size(); i++) order[i] = (int)i;
        for (size_t i = 1; i < order.size(); i++)      /* stable insertion sort by size desc */
          for (size_t j = i; j > 0 && groups[order[j]].size() > groups[order[j-1]].size(); j--)
            std::swap(order[j], order[j-1]);
        std::vector<std::vector<Op>> lanes(team);
        for (int gi : order) {
          int best = 0;
          for (int l = 1; l < team; l++) if (lanes[l].size() < lanes[best].size()) best = l;
          lanes[best].insert(lanes[best].end(), groups[gi].begin(), groups[gi].end());
        }
        for (int l = 0; l < team; l++) {
          start[(size_t)st*team + l] = (int)words.size()/2;
          for (const Op &op : lanes[l]) {
            words.push_back(op.dst | (op.a << 16));
            words.push_back(op.b | (op.k << 16));
          }
        }
      };
      distribute(f, fstart, fops);
      distribute(sv, sstart, sops);
    }
    pivstart[NS] = (int)piv.size();
    fstart[(size_t)NS*team] = (int)fops.size()/2;
    sstart[(size_t)NS*team] = (int)sops.size()/2;
    if (fm->nM >= 65536 || nv >= 65536) { out.error = "model too large for the 16-bit op encoding"; return false; }
    o.st_pivstart = put_i(I, pivstart);
    o.st_piv = put_i(I, piv);
    o.fop_start = put_i(I, fstart);
    while (I.size() % 2) I.push_back(0);
    o.fop = put_i(I, fops);
    o.sop_start = put_i(I, sstart);
    while (I.size() % 2) I.push_back(0);
    o.sop = put_i(I, sops);
  }

  /* collision candidates: plane (static, world frame) vs sphere / capsule end */
  std::vector<int32_t> cbody(nc), ccaps(nc), cbody1(nc, 0);
  std::vector<double> lpos(3*nc), laxis(3*nc), rad(nc), pn(3*nc), pd(nc), cinvw(nc), gquat(4*nc, 0.0);
  m.n_pair = 0;
  m.n_hard = 0;
  bool any_ellipsoid = false;      /* ... or cylinder: candidates whose contact point moves over the geom */
  for (int c = 0; c < nc; c++) {
    int g1 = fm->cand_geom1[c], g2 = fm->cand_geom2[c];
    if (fm->cand_end[c] == 20 || fm->cand_end[c] == 21) {
      /* explicit <pair>, sphere-sphere (mjc_SphereSphere): kind 9.  cand_body / lpos / rad describe
       * geom2 as for a plane candidate; geom1 travels in the plane's slots: cand_body1 = its body,
       * pn = its centre in that body's frame, pd = its radius.  Rows of such a contact live on the
       * chains of TWO bodies: the model runs on the team kernel, whose Newton step takes a dense
       * Hessian while one of them is active (fb_device.h).
       * cand_end 21, a frictionless pair: kind 10, the same geometry; its contact is one hard
       * normal row with a multiplier, which leaves the Hessian tree-sparse. */
      if (fm->geom_type[g1] != FB_GEOM_SPHERE || fm->geom_type[g2] != FB_GEOM_SPHERE ||
          fm->geom_bodyid[g1] < 1 || fm->geom_bodyid[g2] < 1 || fm->geom_bodyid[g1] == fm->geom_bodyid[g2]) {
        out.error = "pair candidates (cand_end 20, 21) must be spheres on two different bodies of the tree"; return false;
      }
      cbody[c] = fm->geom_bodyid[g2]; cbody1[c] = fm->geom_bodyid[g1];
      ccaps[c] = fm->cand_end[c] == 21 ? 10 : 9;
      if (fm->cand_end[c] == 21) m.n_hard++;
      gquat[4*c] = 1.0;
      for (int k = 0; k < 3; k++) { lpos[3*c+k] = fm->geom_pos[3*g2+k]; laxis[3*c+k] = 0.0; pn[3*c+k] = fm->geom_pos[3*g1+k]; }
      rad[c] = fm->geom_size[3*g2];
      pd[c] = fm->geom_size[3*g1];
      cinvw[c] = fm->body_invweight0[2*cbody1[c]] + fm->body_invweight0[2*cbody[c]];
      m.n_pair++;
      continue;
    }
    if (fm->geom_bodyid[g1] != 0 || fm->geom_type[g1] != FB_GEOM_PLANE) {
      out.error = "collision candidates must be world planes vs tree geoms"; return false;
    }
    double pm[9], gm[9];
    quat2mat(fm->geom_quat + 4*g1, pm);
    quat2mat(fm->geom_quat + 4*g2, gm);
    double n[3] = { pm[2], pm[5], pm[8] }, ax[3] = { gm[2], gm[5], gm[8] };
    const int end = fm->cand_end[c];
    cbody[c] = fm->geom_bodyid[g2];
    gquat[4*c] = 1.0;
    if (end == 10) {
      /* ellipsoid (mjc_PlaneConvex): kind 4; lpos = centre, laxis = the three radii, gquat = the
       * geom's orientation in the body frame; rad = the largest radius (conservative checks only) */
      if (fm->geom_type[g2] != FB_GEOM_ELLIPSOID) { out.error = "cand_end 10 on a geom that is not an ellipsoid"; return false; }
      ccaps[c] = 4;
      any_ellipsoid = true;
      const double *sz = fm->geom_size + 3*g2;
      for (int k = 0; k < 3; k++) { lpos[3*c+k] = fm->geom_pos[3*g2+k]; laxis[3*c+k] = sz[k]; pn[3*c+k] = n[k]; }
      rad[c] = std::max(sz[0], std::max(sz[1], sz[2]));
      const double *gq = fm->geom_quat + 4*g2, sgn = gq[0] < 0 ? -1.0 : 1.0;
      for (int k = 0; k < 4; k++) gquat[4*c+k] = sgn*gq[k];
    } else if (end >= 11) {
      /* cylinder (mjc_PlaneCylinder): kinds 5 .. 8 = the lowest rim point, the rim point at the other
       * end, the two triangle points of the lower rim; lpos = centre, laxis = (radius, half length),
       * gquat as for the ellipsoid; rad = the bounding radius (conservative checks only) */
      if (fm->geom_type[g2] != FB_GEOM_CYLINDER) { out.error = "cand_end >= 11 on a geom that is not a cylinder"; return false; }
      ccaps[c] = 5 + (end - 11);
      any_ellipsoid = true;
      const double *sz = fm->geom_size + 3*g2;
      for (int k = 0; k < 3; k++) { lpos[3*c+k] = fm->geom_pos[3*g2+k]; laxis[3*c+k] = k < 2 ? sz[k] : 0.0; pn[3*c+k] = n[k]; }
      rad[c] = std::sqrt(sz[0]*sz[0] + sz[1]*sz[1]);
      const double *gq = fm->geom_quat + 4*g2, sgn = gq[0] < 0 ? -1.0 : 1.0;
      for (int k = 0; k < 4; k++) gquat[4*c+k] = sgn*gq[k];
    } else if (end >= 2) {
      /* box corner end-2 (mjc_PlaneBox): a point of radius 0; kind 2, or 3 for the first corner
       * of its (plane, box) pair; laxis holds the box centre (the corner counts only while it is
       * below the centre along the plane normal) */
      if (fm->geom_type[g2] != FB_GEOM_BOX) { out.error = "cand_end >= 2 on a geom that is not a box"; return false; }
      const int i8 = end - 2;
      const double vec[3] = { (i8 & 1 ? 1 : -1)*fm->geom_size[3*g2], (i8 & 2 ? 1 : -1)*fm->geom_size[3*g2+1],
                              (i8 & 4 ? 1 : -1)*fm->geom_size[3*g2+2] };
      const bool first = c == 0 || fm->cand_geom2[c-1] != g2 || fm->cand_geom1[c-1] != g1;
      ccaps[c] = first ? 3 : 2;
      for (int k = 0; k < 3; k++) {
        lpos[3*c+k] = fm->geom_pos[3*g2+k] + gm[3*k]*vec[0] + gm[3*k+1]*vec[1] + gm[3*k+2]*vec[2];
        laxis[3*c+k] = fm->geom_pos[3*g2+k];
        pn[3*c+k] = n[k];
      }
      rad[c] = 0.0;
    } else {
      if (fm->geom_type[g2] != FB_GEOM_SPHERE && fm->geom_type[g2] != FB_GEOM_CAPSULE) {
        out.error = "collision candidates must be spheres, capsules or boxes"; return false;
      }
      const double off = end*fm->geom_size[3*g2+1];
      ccaps[c] = end != 0;
      for (int k = 0; k < 3; k++) {
        lpos[3*c+k] = fm->geom_pos[3*g2+k] + off*ax[k];
        laxis[3*c+k] = ax[k];
        pn[3*c+k] = n[k];
      }
      rad[c] = fm->geom_size[3*g2];
    }
    pd[c] = n[0]*fm->geom_pos[3*g1] + n[1]*fm->geom_pos[3*g1+1] + n[2]*fm->geom_pos[3*g1+2];
    cinvw[c] = fm->body_invweight0[2*0] + fm->body_invweight0[2*cbody[c]];
  }
  o.cand_body = put_i(I, cbody);
  o.cand_body1 = put_i(I, cbody1);
  o.cand_iscapsule = put_i(I, ccaps);
  o.cand_sensor = put_i(I, ff ? vi(ff->cand_sensor, 4*nc) : std::vector<int32_t>(4*nc, -1));
  o.act_jnt = put_i(I, vi(fm->actuator_trnid, nu));
  o.act_ctrllimited = put_i(I, vi(fm->actuator_ctrllimited, nu));
  o.act_forcelimited = put_i(I, vi(fm->actuator_forcelimited, nu));

  /* farms tables */
  m.n_links = ff ? ff->n_links : 0;
  m.n_joints = ff ? ff->n_joints : 0;
  m.n_contacts = ff ? ff->n_contacts : 0;
  m.n_xfrc = ff ? ff->n_xfrc : 0;
  m.n_swim = ff ? ff->n_swim : 0;
  m.link_cols = ff ? ff->link_cols : 20;
  m.joint_cols = ff ? ff->joint_cols : 18;
  m.contact_cols = ff ? ff->contact_cols : 12;
  m.xfrc_cols = ff ? ff->xfrc_cols : 6;
  if (m.link_cols != 20 || m.contact_cols != 12 || m.xfrc_cols != 6 || m.joint_cols % 2) {
    out.error = "unexpected farms row widths (expected 20 / even / 12 / 6)"; return false;
  }
  m.col_jpos = ff ? ff->col_joint_position : 0;
  m.col_jvel = ff ? ff->col_joint_velocity : 1;
  m.col_jtrq = ff ? ff->col_joint_torque : 11;
  m.col_jlim = ff ? ff->col_joint_limit_force : 16;
  o.link_body = put_i(I, ff ? vi(ff->link_body, m.n_links) : std::vector<int32_t>());
  o.fj_qposadr = put_i(I, ff ? vi(ff->joint_qposadr, m.n_joints) : std::vector<int32_t>());
  o.fj_dofadr = put_i(I, ff ? vi(ff->joint_dofadr, m.n_joints) : std::vector<int32_t>());
  o.fj_jntid = put_i(I, ff ? vi(ff->joint_jntid, m.n_joints) : std::vector<int32_t>());
  o.fj_actpos = put_i(I, ff ? vi(ff->joint_act_position, m.n_joints) : std::vector<int32_t>());
  o.fj_actvel = put_i(I, ff ? vi(ff->joint_act_velocity, m.n_joints) : std::vector<int32_t>());
  o.fj_acttrq = put_i(I, ff ? vi(ff->joint_act_torque, m.n_joints) : std::vector<int32_t>());
  o.xfrc_body = put_i(I, ff ? vi(ff->xfrc_body, m.n_xfrc) : std::vector<int32_t>());
  o.swim_link = put_i(I, ff ? vi(ff->swim_links_index, m.n_swim) : std::vector<int32_t>());
  o.swim_xfrc = put_i(I, ff ? vi(ff->swim_xfrc_index, m.n_swim) : std::vector<int32_t>());
  /* body -> xfrc row (the downstream applier zeroes xfrc_applied, then fills data2xfrc) */
  std::vector<int32_t> body_xfrcrow(nb, -1);
  for (int x = 0; x < m.n_xfrc; x++) {
    int b = ff->xfrc_body[x];
    if (b < 0 || b >= nb) { out.error = "xfrc_body out of range"; return false; }
    body_xfrcrow[b] = x;
  }
  o.body_xfrcrow = put_i(I, body_xfrcrow);
  m.n_wc = wc ? wc->n : 0;
  o.wc_act = put_i(I, wc ? vi(wc->actuator, wc->n) : std::vector<int32_t>());

  /* floats */
  std::vector<double> invw(nb);
  for (int b = 0; b < nb; b++) invw[b] = fm->body_invweight0[2*b];
  o.body_pos = put_f(F, vd(fm->body_pos, 3*nb));
  o.body_quat = put_f(F, vd(fm->body_quat, 4*nb));
  o.body_ipos = put_f(F, vd(fm->body_ipos, 3*nb));
  o.body_iquat = put_f(F, vd(fm->body_iquat, 4*nb));
  o.body_mass = put_f(F, vd(fm->body_mass, nb));
  o.body_inertia = put_f(F, vd(fm->body_inertia, 3*nb));
  o.body_invw = put_f(F, invw);
  o.jnt_pos = put_f(F, vd(fm->jnt_pos, 3*nj));
  o.jnt_axis = put_f(F, vd(fm->jnt_axis, 3*nj));
  o.jnt_stiffness = put_f(F, vd(fm->jnt_stiffness, nj));
  o.jnt_range = put_f(F, vd(fm->jnt_range, 2*nj));
  o.jnt_margin = put_f(F, vd(fm->jnt_margin, nj));
  o.jnt_solref = put_f(F, vd(fm->jnt_solref, 2*nj));
  o.jnt_solimp = put_f(F, vd(fm->jnt_solimp, 5*nj));
  o.jnt_qpos0 = put_f(F, jqpos0);
  o.dof_damping = put_f(F, vd(fm->dof_damping, nv));
  o.dof_armature = put_f(F, vd(fm->dof_armature, nv));
  o.dof_invw = put_f(F, vd(fm->dof_invweight0, nv));
  o.cand_gquat = put_f(F, gquat);
  o.cand_lpos = put_f(F, lpos);
  o.cand_laxis = put_f(F, laxis);
  o.cand_radius = put_f(F, rad);
  o.cand_pn = put_f(F, pn);
  o.cand_pd = put_f(F, pd);
  o.cand_friction = put_f(F, vd(fm->cand_friction, nc));
  o.cand_solref = put_f(F, vd(fm->cand_solref, 2*nc));
  o.cand_solimp = put_f(F, vd(fm->cand_solimp, 5*nc));
  o.cand_margin = put_f(F, vd(fm->cand_margin, nc));
  o.cand_gap = put_f(F, vd(fm->cand_gap, nc));
  o.cand_invw = put_f(F, cinvw);
  std::vector<double> gain(nu);
  for (int a = 0; a < nu; a++) gain[a] = fm->actuator_gainprm[3*a];
  o.act_gain = put_f(F, gain);
  o.act_bias = put_f(F, vd(fm->actuator_biasprm, 3*nu));
  o.act_ctrlrange = put_f(F, vd(fm->actuator_ctrlrange, 2*nu));
  o.act_forcerange = put_f(F, vd(fm->actuator_forcerange, 2*nu));
  o.act_gear = put_f(F, vd(fm->actuator_gear, nu));
  o.swim_mass = put_f(F, ff ? vd(ff->swim_mass, m.n_swim) : std::vector<double>());
  o.swim_height = put_f(F, ff ? vd(ff->swim_height, m.n_swim) : std::vector<double>());
  o.swim_density = put_f(F, ff ? vd(ff->swim_density, m.n_swim) : std::vector<double>());
  o.swim_coef = put_f(F, ff ? vd(ff->swim_coefficients, 6*m.n_swim) : std::vector<double>());
  o.wc_amp = put_f(F, wc ? vd(wc->amplitude, wc->n) : std::vector<double>());
  o.wc_freq = put_f(F, wc ? vd(wc->frequency, wc->n) : std::vector<double>());
  o.wc_lag = put_f(F, wc ? vd(wc->phase_lag, wc->n) : std::vector<double>());
  o.wc_off = put_f(F, wc ? vd(wc->offset, wc->n) : std::vector<double>());
  o.key_qpos = put_f(F, vd(fm->key_qpos, fm->nq));
  o.key_qvel = put_f(F, vd(fm->key_qvel, nv));


  /* ---- environment-per-thread path (fb_fast.h): articulated-body recursion records */
  {
    DevFastLayout &X = m.X;
    X.ok = nb <= FB_FAST_MAXBODY && m.n_pair == 0;    /* two-body rows: not on the per-thread kernels */
    std::vector<FastRec> &rec = out.rec;
    rec.assign(nb, FastRec());
    std::memset(rec.data(), 0, sizeof(FastRec)*nb);
    std::vector<int32_t> actwc(nu > 0 ? nu : 1, -1);
    std::vector<double> chk;
    if (wc) for (int i = 0; i < wc->n; i++) {
      int a = wc->actuator[i];
      if (a < 0 || a >= nu || actwc[a] >= 0) X.ok = 0; else actwc[a] = i;
    }
    int nslot = 0;
    for (int b = 0; b < nb; b++) { rec[b].slot = rec[b].pslot = rec[b].link = rec[b].fj = rec[b].xr = rec[b].swim = -1; rec[b].jtype = -1; rec[b].jid = -1; rec[b].wave_act = -1; }
    for (int b = 1; b < nb; b++) {
      FastRec &r = rec[b];
      int p = fm->body_parentid[b], dn = fm->body_dofnum[b], jid = fm->body_jntid[b];
      int jt = jid >= 0 ? fm->jnt_type[jid] : -1;
      if (!(dn == 0 || (dn == 1 && (jt == FB_JNT_HINGE || jt == FB_JNT_SLIDE)) ||
            (dn == 6 && jt == FB_JNT_FREE && p == 0 && b == 1)))
        X.ok = 0;
      if (dn == 0) jid = -1, jt = -1;
      r.parent = p; r.jtype = jt; r.jid = jid;
      r.pblk = FB_NF*(p - 1);
      r.pblk7 = 7*(p - 1);
      r.qa = jid >= 0 ? fm->jnt_qposadr[jid] : 0;
      r.da = jid >= 0 ? fm->jnt_dofadr[jid] : 0;
      if (jt == FB_JNT_FREE)
        for (int k = 0; k < 6; k++)
          if (fm->dof_damping[r.da + k] != 0 || fm->dof_armature[r.da + k] != 0) X.ok = 0;
      double jp[3] = {0, 0, 0}, pjp[3] = {0, 0, 0};
      if (jid >= 0 && jt != FB_JNT_FREE) for (int k = 0; k < 3; k++) jp[k] = fm->jnt_pos[3*jid + k];
      int pj = fm->body_dofnum[p] > 0 ? fm->body_jntid[p] : -1;
      if (p > 0 && pj >= 0 && fm->jnt_type[pj] != FB_JNT_FREE) for (int k = 0; k < 3; k++) pjp[k] = fm->jnt_pos[3*pj + k];
      for (int k = 0; k < 3; k++) {
        if (jp[k] != 0) r.flags |= FT_HAS_JPOS;
        r.dpos[k] = (float)(fm->body_pos[3*b + k] - pjp[k]);
        r.hloc[k] = (float)(fm->body_ipos[3*b + k] - jp[k]);
        r.jpos[k] = (float)jp[k];
      }
      for (int k = 0; k < 4; k++) r.bquat[k] = (float)fm->body_quat[4*b + k];
      r.mass = (float)fm->body_mass[b];
      /* body inertia about its com in body axes: Riq diag(I) Riq' as xx yy zz xy xz yz */
      double R[9];
      quat2mat(fm->body_iquat + 4*b, R);
      const double *I3 = fm->body_inertia + 3*b;
      auto el = [&](int i, int j) { return R[3*i]*R[3*j]*I3[0] + R[3*i+1]*R[3*j+1]*I3[1] + R[3*i+2]*R[3*j+2]*I3[2]; };
      r.Ib[0] = (float)el(0, 0); r.Ib[1] = (float)el(1, 1); r.Ib[2] = (float)el(2, 2);
      r.Ib[3] = (float)el(0, 1); r.Ib[4] = (float)el(0, 2); r.Ib[5] = (float)el(1, 2);
      /* two equal principal moments: Ia*1 + (Ic - Ia) n n', n the odd principal axis */
      for (int odd = 0; odd < 3; odd++) {
        int e1 = (odd + 1) % 3, e2 = (odd + 2) % 3;
        /* equal up to the rounding of the model compiler (a rotated capsule's two transverse
         * moments differ in the 16th digit), far below what fp32 resolves */
        if (std::fabs(I3[e1] - I3[e2]) <= 1e-10*std::fmax(std::fabs(I3[e1]), std::fabs(I3[e2]))) {
          const double Ia = 0.5*(I3[e1] + I3[e2]);
          r.flags |= FT_AXISYM;
          r.Ib[0] = (float)Ia; r.Ib[1] = (float)(I3[odd] - Ia);
          r.Ib[2] = (float)R[odd]; r.Ib[3] = (float)R[3 + odd]; r.Ib[4] = (float)R[6 + odd]; r.Ib[5] = 0.f;
          break;
        }
      }
      if (p == b - 1) { r.flags |= FT_TO_CARRY; if (p > 0) rec[p].flags |= FT_ADD_CARRY; }
      else if (p > 0 && rec[p].slot < 0) { rec[p].slot = nslot++; rec[p].flags |= FT_HAS_SLOT; }
      if (p != b - 1 && p > 0) r.pslot = rec[p].slot;
      if (jid >= 0 && jt != FB_JNT_FREE) {
        for (int k = 0; k < 3; k++) r.axis[k] = (float)fm->jnt_axis[3*jid + k];
        r.qpos0 = (float)fm->qpos0[r.qa];
        r.margin = (float)fm->jnt_margin[jid];
        r.lo = (float)fm->jnt_range[2*jid]; r.hi = (float)fm->jnt_range[2*jid + 1];
        if (fm->jnt_limited[jid]) r.flags |= FT_LIMITED;
        r.stiffness = (float)fm->jnt_stiffness[jid];
        r.damping = (float)fm->dof_damping[r.da];
        r.armature = (float)fm->dof_armature[r.da];
      }
    }
    /* descending order: the first child to reach a slot stores, the others accumulate */
    {
      std::vector<int> seen(nslot > 0 ? nslot : 1, 0);
      for (int b = nb - 1; b > 0; b--)
        if (rec[b].pslot >= 0 && !seen[rec[b].pslot]) { seen[rec[b].pslot] = 1; rec[b].flags |= FT_FIRST_WRITER; }
    }
    for (int l = 0; l < m.n_links; l++) {
      int b = ff->link_body[l];
      if (b < 1 || b >= nb || rec[b].link >= 0) X.ok = 0; else rec[b].link = l;
    }
    for (int j = 0; j < m.n_joints; j++) {
      int jid = ff->joint_jntid[j];
      /* the row reads qpos/qvel of its own joint and sits on that joint's body */
      if (jid < 0 || jid >= nj || fm->jnt_type[jid] == FB_JNT_FREE || ff->joint_qposadr[j] != fm->jnt_qposadr[jid] ||
          ff->joint_dofadr[j] != fm->jnt_dofadr[jid] || rec[fm->jnt_bodyid[jid]].fj >= 0) { X.ok = 0; continue; }
      rec[fm->jnt_bodyid[jid]].fj = j;
    }
    for (int x = 0; x < m.n_xfrc; x++) {
      int b = ff->xfrc_body[x];
      if (b < 1 || rec[b].xr >= 0) X.ok = 0; else rec[b].xr = x;
    }
    for (int i = 0; i < m.n_swim; i++) {
      int l = ff->swim_links_index[i], xi = ff->swim_xfrc_index[i];
      if (l < 0 || l >= m.n_links || xi < 0 || xi >= m.n_xfrc) { X.ok = 0; continue; }
      int b = ff->link_body[l];
      if (ff->xfrc_body[xi] != b || b < 1 || b >= nb || rec[b].swim >= 0 || rec[b].xr != xi) { X.ok = 0; continue; }
      rec[b].swim = i;
      rec[b].lift = (float)(1000.0*9.81*ff->swim_mass[i]/ff->swim_density[i]);
      if (!(ff->swim_mass[i] > 0)) rec[b].lift = 0.f;
      rec[b].height = (float)ff->swim_height[i];
      for (int k = 0; k < 6; k++) rec[b].coef[k] = (float)ff->swim_coefficients[6*i + k];
    }
    /* actuation: one linear form per joint when nothing clamps, gears are 1 and the farms
     * joint_torque column sums exactly the joint's actuators (physics.py:510-524) */
    std::vector<int32_t> is_off(nu > 0 ? nu : 1, 0);
    for (int b = 1; b < nb; b++) {
      FastRec &r = rec[b];
      if (r.jid < 0 || r.jtype == FB_JNT_FREE) continue;
      bool simple = true;
      int nwave = 0;
      double Kq = 0, Kqd = 0, T0 = 0, KqU = 0, KqdU = 0, T0U = 0;
      for (int a = 0; a < nu; a++) {
        if (fm->actuator_trnid[a] != r.jid) continue;
        /* switched off by initialize_control (task.py:274-286): contributes exactly zero */
        const bool off = fm->actuator_forcelimited[a] && fm->actuator_forcerange[2*a] == 0.0 &&
                         fm->actuator_forcerange[2*a + 1] == 0.0;
        if (off && actwc[a] < 0) { is_off[a] = 1; continue; }
        if (fm->actuator_ctrllimited[a] || fm->actuator_forcelimited[a] || fm->actuator_gear[a] != 1.0) simple = false;
        bool logged = r.fj >= 0 && (ff->joint_act_position[r.fj] == a || ff->joint_act_velocity[r.fj] == a ||
                                    ff->joint_act_torque[r.fj] == a);
        T0 += fm->actuator_biasprm[3*a]; Kq += fm->actuator_biasprm[3*a + 1]; Kqd += fm->actuator_biasprm[3*a + 2];
        if (!logged) {
          T0U += fm->actuator_biasprm[3*a]; KqU += fm->actuator_biasprm[3*a + 1]; KqdU += fm->actuator_biasprm[3*a + 2];
        }
        if (actwc[a] >= 0) {
          int w = actwc[a];
          nwave++;
          if (!logged && r.fj >= 0) simple = false;
          r.wave_act = a;
          r.wgain = (float)fm->actuator_gainprm[3*a];
          r.wamp = (float)wc->amplitude[w]; r.woff = (float)(wc->offset ? wc->offset[w] : 0.0);
          r.wfreq = (float)wc->frequency[w]; r.wlag = (float)wc->phase_lag[w];
        }
      }
      if (nwave > 1) simple = false;
      if (simple) {
        r.flags |= FT_ACT_SIMPLE;
        if (nwave == 1) r.flags |= FT_HAS_WAVE;
        r.Kq = (float)Kq; r.Kqd = (float)Kqd; r.T0 = (float)T0;
        r.KqU = (float)KqU; r.KqdU = (float)KqdU; r.T0U = (float)T0U;
      } else {
        r.wave_act = -1;
      }
    }
    /* conservative plane checks per body: no candidate of the body can be active while
     * n.xpos - pd >= reach, reach = max(|lpos| + radius + margin - gap) over its candidates */
    for (int b = 0; b < nb; b++) {
      rec[b].chk0 = (int)chk.size()/4;
      for (int c = 0; c < nc; c++) {
        if (cbody[c] != b) continue;
        double r = std::sqrt(lpos[3*c]*lpos[3*c] + lpos[3*c+1]*lpos[3*c+1] + lpos[3*c+2]*lpos[3*c+2])
                   + rad[c] + fm->cand_margin[c] - fm->cand_gap[c];
        r *= 1.0 + 1e-5; r += 1e-6;
        bool merged = false;
        for (size_t t = (size_t)rec[b].chk0; t < chk.size()/4; t++)
          if (chk[4*t] == pn[3*c] && chk[4*t+1] == pn[3*c+1] && chk[4*t+2] == pn[3*c+2]) {
            /* same plane normal: keep the larger offset */
            if (pd[c] + r > chk[4*t+3]) chk[4*t+3] = pd[c] + r;
            merged = true;
            break;
          }
        if (!merged) { chk.push_back(pn[3*c]); chk.push_back(pn[3*c+1]); chk.push_back(pn[3*c+2]); chk.push_back(pd[c] + r); }
      }
      rec[b].chk1 = (int)chk.size()/4;
      /* the first check travels in the record; chk0..chk1 are the remaining ones */
      rec[b].chk[0] = rec[b].chk[1] = rec[b].chk[2] = 0.f; rec[b].chk[3] = -1e30f;
      if (rec[b].chk1 > rec[b].chk0) {
        for (int k = 0; k < 4; k++) rec[b].chk[k] = (float)chk[4*(size_t)rec[b].chk0 + k];
        rec[b].chk0++;
      }
    }
    o.ft_actwc = put_i(I, actwc);
    o.ft_actoff = put_i(I, is_off);
    o.ft_chk = put_f(F, chk);
    /* per-thread constrained step: candidates in body order (CandRec), contact sensors as
     * lists of (candidate in that order, sign) */
    {
      std::vector<CandRec> &crec = out.crec;
      crec.clear();
      X.con_ok = X.ok && nc <= FB_FAST_MAXCAND;
      std::vector<int32_t> fc_of(nc > 0 ? nc : 1, -1), sstart(m.n_contacts + 1, 0), scand;
      std::vector<double> ssign;
      for (int b = 0; b < nb; b++) {
        rec[b].bc0 = (int32_t)crec.size();
        for (int c = 0; c < nc; c++) {
          if (cbody[c] != b) continue;
          if (b < 1) { X.con_ok = 0; continue; }
          CandRec r;
          std::memset(&r, 0, sizeof(r));
          r.body = b; r.cid = c; r.iscapsule = ccaps[c]; r.pblk = FB_NF*(b - 1);
          for (int k = 0; k < 3; k++) {
            r.pn[k] = (float)pn[3*c + k];
            r.lpos[k] = (float)(lpos[3*c + k] - (double)rec[b].jpos[k]);
            r.laxis[k] = (float)(ccaps[c] == 2 || ccaps[c] == 3 ? laxis[3*c + k] - (double)rec[b].jpos[k] : laxis[3*c + k]);
          }
          r.mu = (float)fm->cand_friction[c]; r.radius = (float)rad[c]; r.pd = (float)pd[c];
          if (ccaps[c] == 4) {     /* ellipsoid: laxis = radii; the vector part of its orientation (w >= 0) */
            r.radius = (float)gquat[4*c + 1]; r.pad[0] = (float)gquat[4*c + 2]; r.pad[1] = (float)gquat[4*c + 3];
          }
          if (ccaps[c] >= 5) {     /* cylinder point: laxis = the vector part of its orientation; radius, half length */
            for (int k = 0; k < 3; k++) r.laxis[k] = (float)gquat[4*c + 1 + k];
            r.radius = (float)laxis[3*c]; r.pad[0] = (float)laxis[3*c + 1];
          }
          r.includemargin = (float)(fm->cand_margin[c] - fm->cand_gap[c]);
          r.invw = (float)cinvw[c];
          fc_of[c] = (int)crec.size();
          crec.push_back(r);
        }
        rec[b].bc1 = (int32_t)crec.size();
      }
      for (int sx = 0; sx < m.n_contacts; sx++) {
        sstart[sx] = (int)scand.size();
        for (int c = 0; c < nc; c++)
          for (int key = 0; key < 4; key++)
            if (ff->cand_sensor[4*c + key] == sx && fc_of[c] >= 0) { scand.push_back(fc_of[c]); ssign.push_back((key & 1) ? 1.0 : -1.0); }
      }
      sstart[m.n_contacts] = (int)scand.size();
      o.ft_sstart = put_i(I, sstart);
      o.ft_scand = put_i(I, scand);
      o.ft_ssign = put_f(F, ssign);
      X.n_con = NB_NF*(nb - 1) + NR_NF + NC_NF*nc + 6*nslot;
    }
    X.body0 = 0;
    X.slots = FB_NF*(nb - 1);
    X.nslot = nslot;
    X.n_float = X.slots + 27*nslot;
    X.n_scratch = FG_NF*(nb - 1);
    X.n_float_slim = 7*(nb - 1);
    X.n_scratch_slim = (FG_NF + 6)*(nb - 1) + 27*nslot;
    X.jrow_std = m.joint_cols == 18 && m.col_jpos == 0 && m.col_jvel == 1 && m.col_jtrq == 11 && m.col_jlim == 16;
    X.coop_io = fm->nq + nv + (nu > 0 ? nu : 1) + 6*nb <= X.n_float;
    X.coop_io2 = fm->nq + nv + (nu > 0 ? nu : 1) <= X.n_float_slim && 6*nb <= X.n_float_slim;
    {
      std::vector<int> parent(nb);
      for (int b = 0; b < nb; b++) parent[b] = fm->body_parentid[b];
      fb_build_split(parent, X.ok ? FB_SPLIT_MAXW : 1, out.split);
    }
    X.lean = X.ok && X.jrow_std && !any_ellipsoid;      /* (the LEAN constrained kernel leaves the ellipsoid / cylinder branches out) */
    for (int b = 1; b < nb; b++) {
      const FastRec &r = rec[b];
      if (r.flags & FT_HAS_JPOS) X.lean = 0;
      if (!(r.flags & FT_AXISYM)) X.lean = 0;
      if (r.jtype == FB_JNT_SLIDE) X.lean = 0;
      if (r.jtype == FB_JNT_HINGE && !(r.flags & FT_ACT_SIMPLE)) X.lean = 0;
    }
  }

  /* water + units */
  double meters = ff ? ff->meters : 1.0, seconds = ff ? ff->seconds : 1.0,
         kilograms = ff ? ff->kilograms : 1.0;
  double velocity = meters/seconds, accel = meters/(seconds*seconds);
  double newtons = kilograms*accel, torques = kilograms*meters*meters/(seconds*seconds);
  m.inv_meters = (float)(1.0/meters);
  m.inv_velocity = (float)(1.0/velocity);
  m.inv_angvel = (float)seconds;
  m.inv_torques = (float)(1.0/torques);
  m.inv_newtons = (float)(1.0/newtons);
  m.newtons = (float)newtons;
  m.torques = (float)torques;
  m.water_drag = ff ? (ff->water_drag != 0) : 0;
  m.water_buoyancy = ff ? (ff->water_buoyancy != 0) : 0;
  m.water_surface = ff ? (float)ff->water_surface : 0.f;
  m.water_viscosity = ff ? (float)ff->water_viscosity : 1.f;
  for (int k = 0; k < 3; k++) m.water_velocity[k] = ff ? (float)ff->water_velocity[k] : 0.f;

  /* shared-memory layout */
  m.maxcon = nc;
  m.maxefc = 2*nj + 4*nc;
  m.npack = nv*(nv + 1)/2;
  DevLayout &L = m.L;
  int off = 0;
  auto take = [&off](int n) { int r = off; off += (n + 3) & ~3; return r; };
  L.qpos = take(fm->nq); L.qvel = take(nv); L.ctrl = take(nu); L.actf = take(nu);
  L.xpos = take(3*nb); L.xquat = take(4*nb); L.xipos = take(3*nb);
  L.xanchor = take(3*nj); L.xaxis = take(3*nj);
  L.cinert = take(10*nb); L.cdof = take(6*nv); L.cvel = take(6*nb); L.xfrc = take(6*nb);
  L.qM = take(fm->nM); L.qLD = take(fm->nM); L.dinv = take(nv);
  L.fsm = take(nv); L.qacc = take(nv); L.fcon = take(nv); L.grad = take(nv); L.pvec = take(nv);
  L.tmp1 = take(nv); L.tmp2 = take(nv);
  L.limf = take(nj);
  L.scratch = off;
  /* scratch: A = [crb(10nb) | cfrc(6nb)], B = 16nb floats (second buffer of the doubling
   * sums; cacc, buf and the kinematics ping-pong buffer alias into it), see fb_device.h */
  {
    auto pad4 = [](int n) { return (n + 3) & ~3; };
    int nbp = pad4(nb);
    (void)nbp;
    L.crb = L.scratch;
    L.cfrc = L.scratch + 10*nb;
    L.altB = L.scratch + pad4(16*nb);
    L.cacc = L.altB;
    L.buf = L.altB;
    int natural = pad4(16*nb) + pad4(16*nb > 6*nv ? 16*nb : 6*nv);
    int need = 0;   /* the Newton step factors H in M's tree-sparse layout (qLD): no dense scratch */
    L.Md = L.scratch;
    L.H = L.scratch + pad4(m.npack);
    off += natural > need ? natural : need;
  }
  /* models with explicit <pair>s of kind 9: the dense Newton Hessian of the team kernel (nv x nv), a
   * region of its own (the scratch aliases are live during the solve) */
  if (m.n_pair - m.n_hard > 0) L.H = take(nv*nv);
  /* frictionless pairs: the Schur-complement step on their hard normal rows */
  const int nh = m.n_hard;
  L.hV = take(nh*nv); L.hS = take(nh*nh); L.hL = take(nh*nh);
  L.hlam = take(nh); L.hx = take(nh); L.htol = take(nh); L.hrhs = take(nh);
  L.n_float = off;
  L.con_cand = 0;
  L.n_int = (m.maxcon + 3) & ~3;
  L.hcon = L.n_int; L.hon = L.hcon + ((nh + 3) & ~3); L.hws = L.hon + ((nh + 3) & ~3);
  L.n_int = L.hws + ((nh + 3) & ~3);
  if (L.n_int == 0) L.n_int = 4;
  return true;
}

#endif /* FB_MODEL_H_ */
