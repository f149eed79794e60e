/*
 * fb_fastc.h -- the environment-per-thread step WITH joint limits and plane
 * contacts: ONE CUDA thread advances one environment, constraints included.
 *
 * MuJoCo's soft-constraint problem (SURVEY.md A.7/A.8) is the convex programme
 *     min_a  1/2 (a - a0)' M (a - a0) + sum_r s_r(J_r a - aref_r),   s(x) = 1/2 D x^2 [x < 0]
 * whose Newton step solves  H p = -g  with  H = M + J' D_active J.  Every row of J
 * acts on ONE body (a limit on one joint, a plane contact on the touching body),
 * so J' D J is what the mass matrix gains when that body's spatial inertia gains
 *     K_c = X' W X,   W = sum_active D e e'   (e = contact-frame row in world axes,
 *                                              X = velocity of the contact point)
 * and a joint's armature gains D.  H is therefore the joint-space inertia of a tree
 * with augmented bodies, and  H p = -g  is solved WITHOUT forming any matrix by the
 * articulated-body recursion the unconstrained kernel already runs (fb_fast.h):
 * two O(nbody) sweeps per Newton iteration,
 *     A  leaves -> root   the gradient g (see below), articulated inertias with the K_c,
 *                         joint torques = -g
 *     B  root -> leaves   p, J p per row, p . g
 * followed by MuJoCo's exact line search on the piecewise-quadratic cost along p
 * (a safeguarded 1-D Newton iteration over the rows).  The gradient is never
 * assembled from M: with H p = -g, a step a <- a + alpha p changes it to
 *     g' = (1 - alpha) g - J' Delta,   Delta_r = D_r res'_r ([r was active] - [r is active]),
 * i.e. only the rows that SWITCHED contribute, as contact-point forces summed over
 * subtrees by a second (plain) carry of sweep A; p'Mp and p'M(a - a0) of the line search
 * follow from p.g and the row sums at alpha = 0.  J a - aref is carried per row (linear
 * in a).  Neither the mass matrix, nor J, nor a factorisation ever exists: the working
 * set is a few floats per body and per collision candidate, laid out [field][lane] in
 * an L2-resident scratch like the rest of the per-thread state.
 *
 * All environments of a warp walk the same bodies and the same collision
 * CANDIDATES (plane vs sphere / capsule end, fixed by the model; CandRec, in the
 * kernel parameters) with uniform indices.  Whether a candidate touches is a
 * per-lane bit (hm); the warp-wide OR of those bits (hany, one vote per candidate
 * in detect()) lives in uniform registers, so every later loop visits only the
 * candidates SOME lane touches without a memory access or a vote, and the loads of
 * a visited candidate / the next body are issued one visit ahead of their use.
 *
 * The step then is the unconstrained step (fb_fast.h passes 2 and 3: (M + h D) x =
 * f, Euler, log rows, drag) with the constraint forces applied as body wrenches and
 * joint torques, which is MuJoCo's implicit-damping Euler update (SURVEY.md A.10).
 *
 * Reference anchors: mj_step via farms_mujoco/simulation/simulation.py:156; contact
 * aggregation farms_mujoco/sensors/sensors.pyx:20-190; joints rows
 * farms_mujoco/simulation/physics.py:481-524.
 */
#ifndef FB_FASTC_H_
#define FB_FASTC_H_

#include "fb_fast.h"

#ifdef FB_HOST_EMU
/* test harness only: Newton iterations, line-search evaluations, solves (tests/emu) */
static double *fb_emu_stats = 0;
#define FB_FFS(x) __builtin_ffs((int)(x))
#define FB_FFSLL(x) __builtin_ffsll((long long)(x))
#else
#define FB_FFS(x) __ffs((int)(x))
#define FB_FFSLL(x) __ffsll((long long)(x))
#endif

/* LEAN: as in FbFast (hinge joints only, axisymmetric inertias, ...): the unused paths compiled out.
 * SPLIT: as in FbFast -- the 32 environments of a block are stepped by several warps, each owning
 * part of the tree.  Every sweep of the constrained step is a tree sweep with the same two phases
 * (trunk, then the subtrees behind it); a warp's limit rows and collision candidates are those of
 * its own bodies, so its masks (hm, hany, lany) only ever hold its own rows, and the scalars of the
 * line search (row sums, p.g, |p|^2, p'Mp, |a|^2) are summed over the warps through shared memory,
 * in a fixed order, so that every warp of a block takes the same decisions.  The sums are taken in
 * another order than on one warp: results agree with the single-warp kernel to rounding, not bit
 * for bit. */
#define FB_RED_MAX 8       /* values of one cross-warp reduction */
/* ENVP: as in FbFast (per-environment stiffness, damping, drag coefficients, water velocity), and the
 * candidates' friction from the FB_ENV_CAND_FRICTION table where it is set (cand_mu). */
template <int BLK, int LEAN = 0, int SPLIT = 0, int ENVP = 0> struct FbFastCon : FbFast<BLK, 0, LEAN, SPLIT, ENVP> {
  typedef FbFast<BLK, 0, LEAN, SPLIT, ENVP> Base;
  using Base::P; using Base::m; using Base::rec; using Base::s; using Base::env; using Base::gs;
  using Base::cs; using Base::csc; using Base::crec; using Base::hm; using Base::hany;
  using Base::rt; using Base::rootpos; using Base::rqn;
  using Base::block; using Base::gblock; using Base::slot; using Base::nblock; using Base::nroot;
  using Base::ncand;
  using Base::role; using Base::idle; using Base::ord; using Base::ord_n; using Base::ord_bnd;
  unsigned lany[2];      /* bodies whose joint has an active limit row in some lane */
  float *csw;            /* plain-wrench accumulation slots of the branching bodies: 6 floats per slot */
  /* SPLIT: bodies of this warp (bit b), the warps of the block, and the area the warps add their
   * partial sums through: two buffers [warp][FB_RED_MAX][BLK] (lane-offset) used in turn, so that
   * one barrier per reduction is enough */
  unsigned long long own;
  int nroles, red_par;
  float *sred;
  /* The active-set hash of line_eval is linear in the rows' bits, sum_k act_k C^(n-k): the plain sum
   * of the warps' hashes would give rows at the same position of two warps (the two leg pairs of a
   * walker) the same weight, and a foot that lands while its mirror image lifts would leave the sum
   * unchanged.  Each warp's hash is therefore scaled by C^(1024 role) before the sum -- the hash of
   * the warps' row lists laid end to end (a list is shorter than 1024 rows). */
  unsigned hmul;
  FB_MEM int owns(int b) const { return !SPLIT || (int)((own >> b) & 1ull); }
  FB_MEM void con_split_setup(const FastSplit &sp, float *sred_) {
    own = 0ull;
    for (int i = 0; i < ord_n; i++) own |= 1ull << ord[i];
    nroles = sp.nwarps;
    sred = sred_;
    red_par = 0;
    unsigned c1024 = 0x9E3779B1u;
    for (int k = 0; k < 10; k++) c1024 *= c1024;
    hmul = 1u;
    for (int r = 0; r < role; r++) hmul *= c1024;
  }
  /* f[0 .. NF) and u[0 .. NU) <- their sums over the warps of the block, added in warp order by
   * every warp: all warps hold the same bits afterwards and take the same decisions.  Every thread
   * of the block calls it. */
  template <int NF, int NU> FB_MEM void rcombine(float *f, unsigned *u) {
    if (!SPLIT) return;
    float *buf = sred + red_par*(FB_SPLIT_MAXW*FB_RED_MAX*BLK);
    red_par ^= 1;
FB_UNROLL
    for (int k = 0; k < NF; k++) buf[(role*FB_RED_MAX + k)*BLK] = f[k];
FB_UNROLL
    for (int k = 0; k < NU; k++) buf[(role*FB_RED_MAX + NF + k)*BLK] = fb_u2f(u[k]);
    FB_BLOCK_BARRIER();
FB_UNROLL
    for (int k = 0; k < NF; k++) {
      float t = buf[k*BLK];
      for (int r = 1; r < nroles; r++) t += buf[(r*FB_RED_MAX + k)*BLK];
      f[k] = t;
    }
FB_UNROLL
    for (int k = 0; k < NU; k++) {
      unsigned t = fb_f2u(buf[(NF + k)*BLK]);
      for (int r = 1; r < nroles; r++) t += fb_f2u(buf[(r*FB_RED_MAX + NF + k)*BLK]);
      u[k] = t;
    }
  }
  FB_MEM int rany(int flag) {
    unsigned u = flag ? 1u : 0u;
    rcombine<0, 1>(0, &u);
    return u != 0u;
  }
  FB_MEM float *wslot(int i) const { return csw + 6*BLK*i; }

  FB_MEM FbFastCon(const FbParams &P_, const FastRec *rec_, const CandRec *crec_, float *s_, float *gs_,
                   float *cs_, int env_, const FbEnvTables *ept_ = 0)
      : Base(P_, rec_, s_, gs_, env_, ept_) {
    cs = cs_; crec = crec_;
    csc = cs_ + (NB_NF*(P_.m.nbody - 1) + NR_NF)*BLK;
    csw = csc + NC_NF*P_.m.ncand*BLK;
    hm[0] = hm[1] = hany[0] = hany[1] = 0ull;
    lany[0] = lany[1] = 0u;
    own = ~0ull; nroles = 1; red_par = 0; sred = 0; hmul = 1u;
  }

  /* sliding friction of a candidate: ENVP, this environment's where FB_ENV_CAND_FRICTION is set (a
   * uniform null test; the table is indexed by the model's candidate id cid, not the slot).  One load
   * per use site, no copy in the candidate's scratch: so the twins compile without spills, as the
   * kernels without ENVP do. */
  FB_MEM float cand_mu(const CandRec &cr_) const {
    if constexpr (ENVP) {
      const float *fr = this->ept->fric;
      if (fr) return fr[(size_t)cr_.cid*P.env_pad + env];
    }
    return cr_.mu;
  }

  FB_MEM int lane_on(int fc) const { return fb_bit128(hm, fc); }
  FB_MEM int any_on(int fc) const { return fb_bit128(hany, fc); }
  FB_MEM int lim_on(int b) const { return ((b < 32 ? lany[0] : lany[1]) >> (b & 31)) & 1u; }

  /* walk over the set bits of hany in ascending order */
  struct CandIter { int w; unsigned long long mw; };
  FB_MEM CandIter cand_begin() const { CandIter it = {0, hany[0]}; return it; }
  FB_MEM int cand_next(CandIter &it) const {
    if (!it.mw && it.w == 0) { it.w = 1; it.mw = hany[1]; }
    if (!it.mw) return -1;
    const int fc = 64*it.w + FB_FFSLL(it.mw) - 1;
    it.mw &= it.mw - 1;
    return fc;
  }

  /* rotation, com offset and rigid-body inertia of body b about its com (world axes) */
  FB_MEM void body_frame(const FastRec &rc, const float *pb, float *R, float *h, float *Iw) const {
    const Quat q = {pb[(FB_QUAT)*BLK], pb[(FB_QUAT + 1)*BLK], pb[(FB_QUAT + 2)*BLK], pb[(FB_QUAT + 3)*BLK]};
    q_mat(q, R);
    m_rot(R, rc.hloc[0], rc.hloc[1], rc.hloc[2], h);
    if (LEAN || (rc.flags & FT_AXISYM)) {
      float n[3];
      m_rot(R, rc.Ib[2], rc.Ib[3], rc.Ib[4], n);
      const float ia = rc.Ib[0], d0 = rc.Ib[1]*n[0], d1 = rc.Ib[1]*n[1], d2 = rc.Ib[1]*n[2];
      Iw[0] = ia + d0*n[0]; Iw[1] = ia + d1*n[1]; Iw[2] = ia + d2*n[2];
      Iw[3] = d0*n[1]; Iw[4] = d0*n[2]; Iw[5] = d1*n[2];
    } else {
      float T[9];
FB_UNROLL
      for (int i = 0; i < 3; i++) {
        float ri[3] = {R[3*i], R[3*i+1], R[3*i+2]}, t[3];
        sym_mul(rc.Ib, ri, t);
        T[3*i] = t[0]; T[3*i+1] = t[1]; T[3*i+2] = t[2];
      }
      Iw[0] = T[0]*R[0] + T[1]*R[1] + T[2]*R[2];
      Iw[1] = T[3]*R[3] + T[4]*R[4] + T[5]*R[5];
      Iw[2] = T[6]*R[6] + T[7]*R[7] + T[8]*R[8];
      Iw[3] = T[0]*R[3] + T[1]*R[4] + T[2]*R[5];
      Iw[4] = T[0]*R[6] + T[1]*R[7] + T[2]*R[8];
      Iw[5] = T[3]*R[6] + T[4]*R[7] + T[5]*R[8];
    }
  }

  /* ---- limits and plane contacts of the current pose (SURVEY.md A.6/A.7): row parameters
   * into the scratch, masks into registers; NC_RES starts as -aref (n, mu t1, mu t2 parts).
   * Returns 1 when this environment has an active row. */
  FB_MEM int detect() {
    const int nb = m.nbody;
    int mine = 0;
    lany[0] = lany[1] = 0u;
    for (int b = 1; b < nb; b++) {
      const FastRec &rc = rec[b];
      if (!owns(b)) continue;
      if (!(rc.flags & FT_LIMITED) || rc.jtype < 0 || rc.jtype == FB_JNT_FREE) continue;
      const float *pg = gblock(b);
      float *pn = nblock(b);
      const float qj = fb_ld_scr(pg + FG_Q*BLK), qd = fb_ld_scr(pg + FG_QD*BLK);
      const int jid = rc.jid;
      float d2[2] = {0.f, 0.f}, ar2[2] = {0.f, 0.f};
      const float dist2[2] = {qj - rc.lo, rc.hi - qj};
      if (!FB_ANY(dist2[0] < rc.margin || dist2[1] < rc.margin)) continue;
      if (b < 32) lany[0] |= 1u << b; else lany[1] |= 1u << (b - 32);
      float sr[2] = {MF(jnt_solref, 2*jid), MF(jnt_solref, 2*jid + 1)}, si5[5];
      for (int k = 0; k < 5; k++) si5[k] = MF(jnt_solimp, 5*jid + k);
      const float invw = MF(dof_invw, rc.da);
FB_UNROLL
      for (int sd = 0; sd < 2; sd++) {
        if (dist2[sd] < rc.margin) {
          float K, B, imp, R;
          fb_row_params(m.timestep, sr, si5, dist2[sd] - rc.margin, invw, &K, &B, &imp, &R);
          d2[sd] = 1.0f/R;
          /* row Jacobian: +1 (lower), -1 (upper) */
          ar2[sd] = -B*(sd ? -qd : qd) - K*imp*(dist2[sd] - rc.margin);
          mine = 1;
        }
      }
      fb_st_scr(pn + NB_DLO*BLK, d2[0]); fb_st_scr(pn + NB_DHI*BLK, d2[1]);
      fb_st_scr(pn + NB_ARLO*BLK, ar2[0]); fb_st_scr(pn + NB_ARHI*BLK, ar2[1]);
    }
    const float impratio = fmaxf(FB_MINVAL, m.impratio);
    int box_count = 0;           /* corners of the current box that touch (mjc_PlaneBox keeps 4) */
FB_UNROLL
    for (int w = 0; w < 2; w++) {
      unsigned long long mine_w = 0ull, any_w = 0ull;
      const int c1 = m.ncand < 64*w + 64 ? m.ncand : 64*w + 64;
      for (int fc = 64*w; fc < c1; fc++) {
        const CandRec &cr_ = crec[fc];
        if (!owns(cr_.body)) continue;
        const float *pb = s + cr_.pblk*BLK;
        const Quat q = {pb[(FB_QUAT)*BLK], pb[(FB_QUAT + 1)*BLK], pb[(FB_QUAT + 2)*BLK], pb[(FB_QUAT + 3)*BLK]};
        float R[9], t[3], n[3], o[3];
        q_mat(q, R);
        m_rot(R, cr_.lpos[0], cr_.lpos[1], cr_.lpos[2], t);   /* centre - anchor */
FB_UNROLL
        for (int k = 0; k < 3; k++) { n[k] = cr_.pn[k]; o[k] = pb[(FB_ORG + k)*BLK]; }
        const float radius = cr_.radius, includemargin = cr_.includemargin;
        /* plane offset first: both terms are small near the plane */
        const float dist = ((n[0]*rootpos[0] + n[1]*rootpos[1] + n[2]*rootpos[2]) - cr_.pd)
                           + (n[0]*(o[0] + t[0]) + n[1]*(o[1] + t[1]) + n[2]*(o[2] + t[2])) - radius;
        float dist_ = dist, pofs[3] = {0.f, 0.f, 0.f};
        if (!LEAN && cr_.iscapsule == 4) {
          /* ellipsoid (mjc_PlaneConvex): the support point along -normal, R Rg (s o normalize(s o
           * (R Rg)'(-n))), in place of the sphere's -radius n (cr_.radius, pad: the geom's orientation) */
          const float qx = cr_.radius, qy = cr_.pad[0], qz = cr_.pad[1];
          const Quat gq = {sqrtf(fmaxf(0.f, 1.f - qx*qx - qy*qy - qz*qz)), qx, qy, qz};
          float Rg[9], nb_[3], nl[3], w3[3], wb[3];
          q_mat(gq, Rg);
          m_rot_t(R, n[0], n[1], n[2], nb_);
          m_rot_t(Rg, nb_[0], nb_[1], nb_[2], nl);
FB_UNROLL
          for (int k = 0; k < 3; k++) w3[k] = -nl[k]*cr_.laxis[k];
          v_normalize3(w3);
FB_UNROLL
          for (int k = 0; k < 3; k++) w3[k] *= cr_.laxis[k];
          m_rot(Rg, w3[0], w3[1], w3[2], wb);
          m_rot(R, wb[0], wb[1], wb[2], pofs);
          dist_ = ((n[0]*rootpos[0] + n[1]*rootpos[1] + n[2]*rootpos[2]) - cr_.pd)
                  + (n[0]*(o[0] + t[0]) + n[1]*(o[1] + t[1]) + n[2]*(o[2] + t[2])) + (n[0]*pofs[0] + n[1]*pofs[1] + n[2]*pofs[2]);
        }
        if (!LEAN && cr_.iscapsule >= 5) {
          /* cylinder point (mjc_PlaneCylinder): cr_.laxis = the geom's orientation, radius, pad[0] = half length */
          const float qx = cr_.laxis[0], qy = cr_.laxis[1], qz = cr_.laxis[2];
          const Quat gq = {sqrtf(fmaxf(0.f, 1.f - qx*qx - qy*qy - qz*qz)), qx, qy, qz};
          float Rg[9], axis[3], xaxis[3];
          q_mat(gq, Rg);
          m_rot(R, Rg[2], Rg[5], Rg[8], axis);
          m_rot(R, Rg[0], Rg[3], Rg[6], xaxis);
          const float cdist = ((n[0]*rootpos[0] + n[1]*rootpos[1] + n[2]*rootpos[2]) - cr_.pd)
                              + (n[0]*(o[0] + t[0]) + n[1]*(o[1] + t[1]) + n[2]*(o[2] + t[2]));
          dist_ = fb_plane_cylinder_point(n, axis, xaxis, cr_.radius, cr_.pad[0], cr_.iscapsule - 5, cdist, pofs);
        }
        const int ell = !LEAN && cr_.iscapsule >= 4;       /* the contact point moves over the geom: dist_, pofs */
        int hit = (ell ? dist_ : dist) < includemargin;
        if ((cr_.iscapsule & ~1) == 2) {
          /* box corner: only while it is below the box centre along the normal, at most 4 per box */
          float u[3];
          m_rot(R, cr_.lpos[0] - cr_.laxis[0], cr_.lpos[1] - cr_.laxis[1], cr_.lpos[2] - cr_.laxis[2], u);
          if (cr_.iscapsule == 3) box_count = 0;
          if (n[0]*u[0] + n[1]*u[1] + n[2]*u[2] > 0.f || box_count >= 4) hit = 0;
          box_count += hit;
        }
        if (!FB_ANY(hit)) continue;
        any_w |= 1ull << (fc & 63);
        if (hit) mine_w |= 1ull << (fc & 63);
        float *pc = ncand(fc);
        float r[3], f[9];
FB_UNROLL
        for (int k = 0; k < 3; k++) { r[k] = ell ? t[k] + pofs[k] - n[k]*(0.5f*dist_) : t[k] - n[k]*(radius + 0.5f*dist); f[k] = n[k]; }
        const float de = ell ? dist_ : dist;
        if (cr_.iscapsule == 1) m_rot(R, cr_.laxis[0], cr_.laxis[1], cr_.laxis[2], f + 3);
        else f[3] = f[4] = f[5] = 0.f;
        /* mju_makeFrame */
        v_normalize3(f);
        if (sqrtf(f[3]*f[3] + f[4]*f[4] + f[5]*f[5]) < 0.5f) {
          f[3] = f[4] = f[5] = 0.f;
          if (f[1] < 0.5f && f[1] > -0.5f) f[4] = 1.f; else f[5] = 1.f;
        }
        const float dt = f[0]*f[3] + f[1]*f[4] + f[2]*f[5];
        f[3] -= dt*f[0]; f[4] -= dt*f[1]; f[5] -= dt*f[2];
        v_normalize3(f + 3);
        v_cross(f, f + 3, f + 6);
        const float mu = cand_mu(cr_);
        const int c = cr_.cid;
        float sr[2] = {MF(cand_solref, 2*c), MF(cand_solref, 2*c + 1)}, si5[5];
        for (int k = 0; k < 5; k++) si5[k] = MF(cand_solimp, 5*c + k);
        const float tran = cr_.invw;
        float K, B, imp, Rr;
        fb_row_params(m.timestep, sr, si5, de - includemargin, tran + mu*mu*tran, &K, &B, &imp, &Rr);
        const float R1 = Rr/impratio;
        const float cmu2 = mu*mu*(R1/Rr);
        const float Rpy = fmaxf(FB_MINVAL, 2.f*cmu2*R1);
        /* velocity of the contact point */
        float vp[3], cr[3];
        const float wv[3] = {pb[(FB_VEL)*BLK], pb[(FB_VEL + 1)*BLK], pb[(FB_VEL + 2)*BLK]};
        v_cross(wv, r, cr);
FB_UNROLL
        for (int k = 0; k < 3; k++) vp[k] = pb[(FB_VEL + 3 + k)*BLK] + cr[k];
        const float vn = f[0]*vp[0] + f[1]*vp[1] + f[2]*vp[2];
        const float vt1 = f[3]*vp[0] + f[4]*vp[1] + f[5]*vp[2];
        const float vt2 = f[6]*vp[0] + f[7]*vp[1] + f[8]*vp[2];
        /* aref of the four pyramid rows = base +- bt1, base +- bt2 */
        const float base = -B*vn - K*imp*(de - includemargin);
FB_UNROLL
        for (int k = 0; k < 3; k++) { fb_st_scr(pc + (NC_R + k)*BLK, r[k]); fb_st_scr(pc + (NC_T1 + k)*BLK, f[3 + k]); }
        fb_st_scr(pc + NC_D*BLK, hit ? 1.0f/Rpy : 0.f);
        fb_st_scr(pc + (NC_RES)*BLK, -base);
        fb_st_scr(pc + (NC_RES + 1)*BLK, B*mu*vt1);
        fb_st_scr(pc + (NC_RES + 2)*BLK, B*mu*vt2);
        mine |= hit;
      }
      hm[w] = mine_w; hany[w] = any_w;
    }
    return mine;
  }

  /* pure J a of a candidate's rows from the body's pure spatial acceleration al (about the
   * anchor): (n, mu t1, mu t2) . (al_lin + al_ang x r) */
  FB_MEM void rows_of(int fc, const float *pc, const float *al, float *out) const {
    const CandRec &cr_ = crec[fc];
    float n[3] = {cr_.pn[0], cr_.pn[1], cr_.pn[2]}, t1[3], t2[3], r[3], cr[3], pa[3];
FB_UNROLL
    for (int k = 0; k < 3; k++) { t1[k] = fb_ld_scr(pc + (NC_T1 + k)*BLK); r[k] = fb_ld_scr(pc + (NC_R + k)*BLK); }
    v_cross(n, t1, t2);
    v_cross(al, r, cr);
FB_UNROLL
    for (int k = 0; k < 3; k++) pa[k] = al[3 + k] + cr[k];
    const float mu = cand_mu(cr_);
    out[0] = n[0]*pa[0] + n[1]*pa[1] + n[2]*pa[2];
    out[1] = mu*(t1[0]*pa[0] + t1[1]*pa[1] + t1[2]*pa[2]);
    out[2] = mu*(t2[0]*pa[0] + t2[1]*pa[1] + t2[2]*pa[2]);
  }

  /* ---- root -> leaves after pass_inertia_m<1>: the unconstrained acceleration a0 (joint
   * space, classical MuJoCo qacc), and J a0 - aref of every candidate row.  Two carries: the
   * spatial acceleration with its velocity-product terms (what the recursion needs) and the
   * pure J a part (what the rows see). */
  FB_MEM void smooth_accel(const float *aroot) {
    const int nb = m.nbody;
    float ac[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, lc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float nx[9];      /* U[6], u, 1/d, qd of the next body to visit */
    const int n_it = SPLIT ? ord_n : nb - 1;
    {
      const int b0 = SPLIT ? (ord_n > 0 ? ord[0] : 1) : 1;
      const float *pn = nblock(b0);
FB_UNROLL
      for (int k = 0; k < 8; k++) nx[k] = fb_ld_scr(pn + (NB_U + k)*BLK);
      nx[8] = fb_ld_scr(gblock(b0) + FG_QD*BLK);
    }
    for (int i = 0; i <= n_it; i++) {
      if (SPLIT && i == ord_bnd) this->split_barrier();      /* the trunk's accelerations are known */
      if (i == n_it) break;
      const int b = SPLIT ? ord[i] : i + 1;
      const int bn = SPLIT ? (i + 1 < n_it ? ord[i + 1] : 0) : (i + 2 < nb ? i + 2 : 0);
      const FastRec &rc = rec[b];
      const float *pb = block(b);
      float *pn = nblock(b);
      const int jtype = rc.jtype, flags = rc.flags;
      float cx[9];
FB_UNROLL
      for (int k = 0; k < 9; k++) cx[k] = nx[k];
      if (bn) {
        const float *pn1 = nblock(bn);
FB_UNROLL
        for (int k = 0; k < 8; k++) nx[k] = fb_ld_scr(pn1 + (NB_U + k)*BLK);
        nx[8] = fb_ld_scr(gblock(bn) + FG_QD*BLK);
      }
      const Quat q = {pb[(FB_QUAT)*BLK], pb[(FB_QUAT + 1)*BLK], pb[(FB_QUAT + 2)*BLK], pb[(FB_QUAT + 3)*BLK]};
      float R[9], v[6], a[6], al[6];
      q_mat(q, R);
FB_UNROLL
      for (int k = 0; k < 6; k++) v[k] = pb[(FB_VEL + k)*BLK];
      if (jtype == FB_JNT_FREE) {
        float cr[3];
        v_cross(v, v + 3, cr);
        float *pr = nroot();
FB_UNROLL
        for (int k = 0; k < 3; k++) {
          a[k] = aroot[k]; a[3 + k] = aroot[3 + k];
          al[k] = aroot[k]; al[3 + k] = aroot[3 + k] + m.grav[k] + cr[k];
        }
FB_UNROLL
        for (int k = 0; k < 6; k++) { fb_st_scr(pr + (NR_A + k)*BLK, al[k]); fb_st_scr(pr + (NR_MD + k)*BLK, 0.f); }
      } else {
        float ap[6] = {0.f, 0.f, 0.f, -m.grav[0], -m.grav[1], -m.grav[2]}, lp[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        float r[3] = {0.f, 0.f, 0.f}, cr[3];
        if (rc.parent > 0) {
          const float *pp = (s + rc.pblk*BLK);
FB_UNROLL
          for (int k = 0; k < 3; k++) r[k] = pb[(FB_ORG + k)*BLK] - pp[(FB_ORG + k)*BLK];
          if (flags & FT_TO_CARRY) {
FB_UNROLL
            for (int k = 0; k < 6; k++) { ap[k] = ac[k]; lp[k] = lc[k]; }
          } else {
            const float *so = slot(rc.pslot);
FB_UNROLL
            for (int k = 0; k < 6; k++) { ap[k] = so[k*BLK]; lp[k] = so[(6 + k)*BLK]; }
          }
        }
        v_cross(ap, r, cr);
FB_UNROLL
        for (int k = 0; k < 3; k++) { a[k] = ap[k]; a[3 + k] = ap[3 + k] + cr[k]; }
        v_cross(lp, r, cr);
FB_UNROLL
        for (int k = 0; k < 3; k++) { al[k] = lp[k]; al[3 + k] = lp[3 + k] + cr[k]; }
        if (jtype >= 0) {
          const float qd = cx[8];
          float ax[3];
          m_rot(R, rc.axis[0], rc.axis[1], rc.axis[2], ax);
          const float *U = cx;
          float aq[3] = {ax[0]*qd, ax[1]*qd, ax[2]*qd}, c[3];
          if (LEAN || jtype == FB_JNT_HINGE) {
            v_cross(v, aq, c);
            a[0] += c[0]; a[1] += c[1]; a[2] += c[2];
            v_cross(v + 3, aq, c);
            a[3] += c[0]; a[4] += c[1]; a[5] += c[2];
          } else {
            v_cross(v, aq, c);
            a[3] += c[0]; a[4] += c[1]; a[5] += c[2];
          }
          const float ua = U[0]*a[0] + U[1]*a[1] + U[2]*a[2] + U[3]*a[3] + U[4]*a[4] + U[5]*a[5];
          const float qdd = (cx[7] - ua)*cx[6];
          if (LEAN || jtype == FB_JNT_HINGE) {
FB_UNROLL
            for (int k = 0; k < 3; k++) { a[k] += ax[k]*qdd; al[k] += ax[k]*qdd; }
          } else {
FB_UNROLL
            for (int k = 0; k < 3; k++) { a[3 + k] += ax[k]*qdd; al[3 + k] += ax[k]*qdd; }
          }
          fb_st_scr(pn + NB_A*BLK, qdd);
          fb_st_scr(pn + NB_MD*BLK, 0.f);
        }
      }
FB_UNROLL
      for (int k = 0; k < 6; k++) { ac[k] = a[k]; lc[k] = al[k]; }
      if (flags & FT_HAS_SLOT) {
        float *so = slot(rc.slot);
FB_UNROLL
        for (int k = 0; k < 6; k++) { so[k*BLK] = a[k]; so[(6 + k)*BLK] = al[k]; }
      }
      for (int fc = rc.bc0; fc < rc.bc1; fc++) {
        if (!any_on(fc)) continue;
        float *pc = ncand(fc);
        float ja[3];
        rows_of(fc, pc, al, ja);
FB_UNROLL
        for (int k = 0; k < 3; k++) fb_st_scr(pc + (NC_RES + k)*BLK, fb_ld_scr(pc + (NC_RES + k)*BLK) + ja[k]);
      }
    }
  }

  /* ---- Newton sweep A: leaves -> root.  Articulated inertias of the augmented tree, U, u, 1/d
   * per joint; the floating root's p */
  FB_MEM void newton_a(float keep) {
    const int nb = m.nbody;
    ArtInertia C;
    float pc6[6], wc[6];     /* carries from child b+1: articulated bias, plain wrench of the switched rows */
FB_UNROLL
    for (int k = 0; k < 6; k++) { C.A[k] = 0.f; C.M[k] = 0.f; pc6[k] = 0.f; wc[k] = 0.f; }
FB_UNROLL
    for (int k = 0; k < 9; k++) C.H[k] = 0.f;
    float nx[2];      /* previous gradient entry, a of the next joint to visit */
    const int n_it = SPLIT ? ord_n : nb - 1;
    {
      const int b0 = SPLIT ? (ord_n > 0 ? ord[ord_n - 1] : 1) : nb - 1;
      nx[0] = fb_ld_scr(nblock(b0) + NB_MD*BLK); nx[1] = fb_ld_scr(nblock(b0) + NB_A*BLK);
    }
    for (int i = n_it; i >= 0; i--) {
      if (SPLIT && i == ord_bnd) this->split_barrier();      /* the subtrees have handed over: the trunk goes on */
      if (i == 0) break;
      const int b = SPLIT ? ord[i - 1] : i;
      const int bn = SPLIT ? (i >= 2 ? ord[i - 2] : 0) : (i > 1 ? i - 1 : 0);
      const FastRec &rc = rec[b];
      FB_PIN_I(rc.jtype); FB_PIN_I(rc.flags); FB_PIN_I(rc.pblk); FB_PIN_I(rc.parent); FB_PIN_I(rc.bc0); FB_PIN_I(rc.bc1);
      FB_PIN_F(rc.mass); FB_PIN_F(rc.armature);
FB_UNROLL
      for (int k = 0; k < 3; k++) { FB_PIN_F(rc.hloc[k]); FB_PIN_F(rc.axis[k]); }
FB_UNROLL
      for (int k = 0; k < 5; k++) FB_PIN_F(rc.Ib[k]);
      const float *pb = block(b);
      float *pn = nblock(b);
      const int jtype = rc.jtype, flags = rc.flags;
      const float md = nx[0], aj = nx[1];
      if (bn) { nx[0] = fb_ld_scr(nblock(bn) + NB_MD*BLK); nx[1] = fb_ld_scr(nblock(bn) + NB_A*BLK); }
      float lim4[4] = {0.f, 0.f, 0.f, 0.f}, dtau = 0.f;
      const int limited = (flags & FT_LIMITED) && lim_on(b);
      if (limited) {
FB_UNROLL
        for (int k = 0; k < 4; k++) lim4[k] = fb_ld_scr(pn + (NB_DLO + k)*BLK);
        dtau = fb_ld_scr(pn + NB_MP*BLK);
      }
      float R[9], h[3], Iw[6], pA[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, W[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      body_frame(rc, pb, R, h, Iw);
      const float mass = rc.mass;
      ArtInertia I;
      const float hh = h[0]*h[0] + h[1]*h[1] + h[2]*h[2];
      I.A[0] = Iw[0] + mass*(hh - h[0]*h[0]); I.A[1] = Iw[1] + mass*(hh - h[1]*h[1]);
      I.A[2] = Iw[2] + mass*(hh - h[2]*h[2]);
      I.A[3] = Iw[3] - mass*h[0]*h[1]; I.A[4] = Iw[4] - mass*h[0]*h[2]; I.A[5] = Iw[5] - mass*h[1]*h[2];
      I.H[0] = 0.f; I.H[1] = -mass*h[2]; I.H[2] = mass*h[1];
      I.H[3] = mass*h[2]; I.H[4] = 0.f; I.H[5] = -mass*h[0];
      I.H[6] = -mass*h[1]; I.H[7] = mass*h[0]; I.H[8] = 0.f;
      I.M[0] = mass; I.M[1] = mass; I.M[2] = mass; I.M[3] = 0.f; I.M[4] = 0.f; I.M[5] = 0.f;
      /* active contact rows of this body: K_c; switched rows: their force */
      for (int fc = rc.bc0; fc < rc.bc1; fc++) {
        if (!any_on(fc)) continue;
        const CandRec &cr_ = crec[fc];
        const float *pc = ncand(fc);
        const int on = lane_on(fc);
        const float D = on ? fb_ld_scr(pc + NC_D*BLK) : 0.f;
        const float dn = on ? fb_ld_scr(pc + NC_JP*BLK) : 0.f, d1 = on ? fb_ld_scr(pc + (NC_JP + 1)*BLK) : 0.f,
                    d2 = on ? fb_ld_scr(pc + (NC_JP + 2)*BLK) : 0.f;
        const float rn = fb_ld_scr(pc + NC_RES*BLK), r1 = fb_ld_scr(pc + (NC_RES + 1)*BLK), r2 = fb_ld_scr(pc + (NC_RES + 2)*BLK);
        float n[3] = {cr_.pn[0], cr_.pn[1], cr_.pn[2]}, t1[3], t2[3], r[3];
FB_UNROLL
        for (int k = 0; k < 3; k++) { t1[k] = fb_ld_scr(pc + (NC_T1 + k)*BLK); r[k] = fb_ld_scr(pc + (NC_R + k)*BLK); }
        v_cross(n, t1, t2);
        const float mu = cand_mu(cr_);
        ArtInertia Kc;
        float p6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
FB_UNROLL
        for (int k = 0; k < 6; k++) { Kc.A[k] = 0.f; Kc.M[k] = 0.f; }
FB_UNROLL
        for (int k = 0; k < 9; k++) Kc.H[k] = 0.f;
FB_UNROLL
        for (int row = 0; row < 4; row++) {
          const float sg = (row & 1) ? -1.f : 1.f;
          const float res = rn + sg*(row < 2 ? r1 : r2);
          const float w = (D > 0.f && res < 0.f) ? D : 0.f;
          const float e0 = n[0] + sg*mu*(row < 2 ? t1[0] : t2[0]);
          const float e1 = n[1] + sg*mu*(row < 2 ? t1[1] : t2[1]);
          const float e2 = n[2] + sg*mu*(row < 2 ? t1[2] : t2[2]);
          const float w0 = w*e0, w1 = w*e1, w2 = w*e2;
          Kc.M[0] += w0*e0; Kc.M[1] += w1*e1; Kc.M[2] += w2*e2;
          Kc.M[3] += w0*e1; Kc.M[4] += w0*e2; Kc.M[5] += w1*e2;
        }
        art_shift(Kc, p6, r);
FB_UNROLL
        for (int k = 0; k < 6; k++) { I.A[k] += Kc.A[k]; I.M[k] += Kc.M[k]; }
FB_UNROLL
        for (int k = 0; k < 9; k++) I.H[k] += Kc.H[k];
        {
          const float Fd[3] = {dn*n[0] + d1*t1[0] + d2*t2[0], dn*n[1] + d1*t1[1] + d2*t2[1],
                               dn*n[2] + d1*t1[2] + d2*t2[2]};
          float cr[3];
          v_cross(r, Fd, cr);
FB_UNROLL
          for (int k = 0; k < 3; k++) { W[k] += cr[k]; W[3 + k] += Fd[k]; }
        }
      }
      if (flags & FT_ADD_CARRY) {
FB_UNROLL
        for (int k = 0; k < 6; k++) { I.A[k] += C.A[k]; I.M[k] += C.M[k]; pA[k] += pc6[k]; W[k] += wc[k]; }
FB_UNROLL
        for (int k = 0; k < 9; k++) I.H[k] += C.H[k];
      }
      if (flags & FT_HAS_SLOT) {
        const float *so = slot(rc.slot);
        const float *sw = wslot(rc.slot);
FB_UNROLL
        for (int k = 0; k < 6; k++) {
          I.A[k] += so[k*BLK]; I.M[k] += so[(15 + k)*BLK]; pA[k] += so[(21 + k)*BLK];
          W[k] += fb_ld_scr(sw + k*BLK);
        }
FB_UNROLL
        for (int k = 0; k < 9; k++) I.H[k] += so[(6 + k)*BLK];
      }
      if (jtype == FB_JNT_FREE) {
        float K[6][6], rhs[6], x[6];
        float *pr = nroot();
        K[0][0] = I.A[0]; K[1][1] = I.A[1]; K[2][2] = I.A[2];
        K[1][0] = I.A[3]; K[2][0] = I.A[4]; K[2][1] = I.A[5];
        K[3][3] = I.M[0]; K[4][4] = I.M[1]; K[5][5] = I.M[2];
        K[4][3] = I.M[3]; K[5][3] = I.M[4]; K[5][4] = I.M[5];
FB_UNROLL
        for (int i = 0; i < 3; i++)
FB_UNROLL
          for (int j = 0; j < 3; j++) K[3 + j][i] = I.H[3*i + j];
FB_UNROLL
        for (int k = 0; k < 6; k++) {
          const float g = keep*fb_ld_scr(pr + (NR_MD + k)*BLK) - W[k];
          fb_st_scr(pr + (NR_MD + k)*BLK, g);
          rhs[k] = -pA[k] - g;
        }
        solve6(K, rhs, x);
FB_UNROLL
        for (int k = 0; k < 6; k++) fb_st_scr(pr + (NR_P + k)*BLK, x[k]);
        continue;
      }
      if (jtype >= 0) {
        float ax[3], U[6], d, u;
        m_rot(R, rc.axis[0], rc.axis[1], rc.axis[2], ax);
        /* gradient entry of this joint: what is left of the previous one, minus the switched rows */
        const float g = keep*md - dtau - ((LEAN || jtype == FB_JNT_HINGE) ? ax[0]*W[0] + ax[1]*W[1] + ax[2]*W[2]
                                                                 : ax[0]*W[3] + ax[1]*W[4] + ax[2]*W[5]);
        fb_st_scr(pn + NB_MD*BLK, g);
        const float tau = -g;
        float dl = 0.f;
        if (limited) {
          const float rlo = aj - lim4[2], rhi = -aj - lim4[3];
          if (lim4[0] > 0.f && rlo < 0.f) dl += lim4[0];
          if (lim4[1] > 0.f && rhi < 0.f) dl += lim4[1];
        }
        if (LEAN || jtype == FB_JNT_HINGE) {
          sym_mul(I.A, ax, U);
          ht_mul(I.H, ax, U + 3);
          d = ax[0]*U[0] + ax[1]*U[1] + ax[2]*U[2];
          u = tau - (ax[0]*pA[0] + ax[1]*pA[1] + ax[2]*pA[2]);
        } else {
          h_mul(I.H, ax, U);
          sym_mul(I.M, ax, U + 3);
          d = ax[0]*U[3] + ax[1]*U[4] + ax[2]*U[5];
          u = tau - (ax[0]*pA[3] + ax[1]*pA[4] + ax[2]*pA[5]);
        }
        d += rc.armature + dl;
        const float dinv = fb_rcp(d);
        sym_rank1(I.A, U, dinv);
        sym_rank1(I.M, U + 3, dinv);
FB_UNROLL
        for (int i = 0; i < 3; i++) {
          const float ui = dinv*U[i];
FB_UNROLL
          for (int j = 0; j < 3; j++) I.H[3*i + j] -= ui*U[3 + j];
        }
        const float ud = u*dinv;
FB_UNROLL
        for (int k = 0; k < 6; k++) { pA[k] += U[k]*ud; fb_st_scr(pn + (NB_U + k)*BLK, U[k]); }
        fb_st_scr(pn + NB_DINV*BLK, dinv); fb_st_scr(pn + NB_UU*BLK, u);
      }
      if (rc.parent == 0) continue;
      {
        const float *pp = (s + rc.pblk*BLK);
        float r[3];
FB_UNROLL
        for (int k = 0; k < 3; k++) r[k] = pb[(FB_ORG + k)*BLK] - pp[(FB_ORG + k)*BLK];
        art_shift(I, pA, r);
        float cr[3];
        v_cross(r, W + 3, cr);
        W[0] += cr[0]; W[1] += cr[1]; W[2] += cr[2];
      }
      if (flags & FT_TO_CARRY) {
        C = I;
FB_UNROLL
        for (int k = 0; k < 6; k++) { pc6[k] = pA[k]; wc[k] = W[k]; }
      } else {
        float *so = slot(rc.pslot);
        float *sw = wslot(rc.pslot);
        if (flags & FT_FIRST_WRITER) {
FB_UNROLL
          for (int k = 0; k < 6; k++) {
            so[k*BLK] = I.A[k]; so[(15 + k)*BLK] = I.M[k]; so[(21 + k)*BLK] = pA[k];
            fb_st_scr(sw + k*BLK, W[k]);
          }
FB_UNROLL
          for (int k = 0; k < 9; k++) so[(6 + k)*BLK] = I.H[k];
        } else {
FB_UNROLL
          for (int k = 0; k < 6; k++) {
            so[k*BLK] += I.A[k]; so[(15 + k)*BLK] += I.M[k]; so[(21 + k)*BLK] += pA[k];
            fb_st_scr(sw + k*BLK, fb_ld_scr(sw + k*BLK) + W[k]);
          }
FB_UNROLL
          for (int k = 0; k < 9; k++) so[(6 + k)*BLK] += I.H[k];
        }
      }
    }
  }

  /* ---- Newton sweep B: root -> leaves.  p per joint, the bodies' pure accelerations, J p per
   * candidate row; g0 = p . g, pp = |p|^2 */
  FB_MEM void newton_b(float *g0_out, float *pp_out, int store_ap) {
    const int nb = m.nbody;
    float lc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float g0 = 0.f, pp = 0.f;
    float nx[9];      /* U[6], 1/d, u, gradient entry of the next body to visit */
    const int n_it = SPLIT ? ord_n : nb - 1;
    {
      const float *pn = nblock(SPLIT ? (ord_n > 0 ? ord[0] : 1) : 1);
FB_UNROLL
      for (int k = 0; k < 8; k++) nx[k] = fb_ld_scr(pn + (NB_U + k)*BLK);
      nx[8] = fb_ld_scr(pn + NB_MD*BLK);
    }
    for (int i = 0; i <= n_it; i++) {
      if (SPLIT && i == ord_bnd) this->split_barrier();      /* the trunk's p is known */
      if (i == n_it) break;
      const int b = SPLIT ? ord[i] : i + 1;
      const int bn = SPLIT ? (i + 1 < n_it ? ord[i + 1] : 0) : (i + 2 < nb ? i + 2 : 0);
      const FastRec &rc = rec[b];
      FB_PIN_I(rc.jtype); FB_PIN_I(rc.flags); FB_PIN_I(rc.pblk); FB_PIN_I(rc.parent); FB_PIN_I(rc.bc0); FB_PIN_I(rc.bc1);
FB_UNROLL
      for (int k = 0; k < 3; k++) FB_PIN_F(rc.axis[k]);
      const float *pb = block(b);
      float *pn = nblock(b);
      const int jtype = rc.jtype, flags = rc.flags;
      float cx[9];
FB_UNROLL
      for (int k = 0; k < 9; k++) cx[k] = nx[k];
      if (bn) {
        const float *pn1 = nblock(bn);
FB_UNROLL
        for (int k = 0; k < 8; k++) nx[k] = fb_ld_scr(pn1 + (NB_U + k)*BLK);
        nx[8] = fb_ld_scr(pn1 + NB_MD*BLK);
      }
      float al[6];
      if (jtype == FB_JNT_FREE) {
        const float *pr = nroot();
FB_UNROLL
        for (int k = 0; k < 6; k++) {
          al[k] = fb_ld_scr(pr + (NR_P + k)*BLK);
          g0 += al[k]*fb_ld_scr(pr + (NR_MD + k)*BLK);
          pp += al[k]*al[k];
        }
      } else {
        float lp[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, r[3] = {0.f, 0.f, 0.f}, cr[3];
        if (rc.parent > 0) {
          const float *pp_ = (s + rc.pblk*BLK);
FB_UNROLL
          for (int k = 0; k < 3; k++) r[k] = pb[(FB_ORG + k)*BLK] - pp_[(FB_ORG + k)*BLK];
          if (flags & FT_TO_CARRY) {
FB_UNROLL
            for (int k = 0; k < 6; k++) lp[k] = lc[k];
          } else {
            const float *so = slot(rc.pslot);
FB_UNROLL
            for (int k = 0; k < 6; k++) lp[k] = so[k*BLK];
          }
        }
        v_cross(lp, r, cr);
FB_UNROLL
        for (int k = 0; k < 3; k++) { al[k] = lp[k]; al[3 + k] = lp[3 + k] + cr[k]; }
        if (jtype >= 0) {
          const Quat q = {pb[(FB_QUAT)*BLK], pb[(FB_QUAT + 1)*BLK], pb[(FB_QUAT + 2)*BLK], pb[(FB_QUAT + 3)*BLK]};
          float R[9], ax[3];
          q_mat(q, R);
          m_rot(R, rc.axis[0], rc.axis[1], rc.axis[2], ax);
          const float *U = cx;
          const float ua = U[0]*al[0] + U[1]*al[1] + U[2]*al[2] + U[3]*al[3] + U[4]*al[4] + U[5]*al[5];
          const float pj = (cx[7] - ua)*cx[6];
          if (LEAN || jtype == FB_JNT_HINGE) { al[0] += ax[0]*pj; al[1] += ax[1]*pj; al[2] += ax[2]*pj; }
          else { al[3] += ax[0]*pj; al[4] += ax[1]*pj; al[5] += ax[2]*pj; }
          fb_st_scr(pn + NB_P*BLK, pj); g0 += pj*cx[8];
          pp += pj*pj;
        }
      }
FB_UNROLL
      for (int k = 0; k < 6; k++) lc[k] = al[k];
      if (store_ap) {
FB_UNROLL
        for (int k = 0; k < 6; k++) fb_st_scr(pn + (NB_AP + k)*BLK, al[k]);
      }
      if (flags & FT_HAS_SLOT) {
        float *so = slot(rc.slot);
FB_UNROLL
        for (int k = 0; k < 6; k++) so[k*BLK] = al[k];
      }
      for (int fc = rc.bc0; fc < rc.bc1; fc++) {
        if (!any_on(fc)) continue;
        float *pc = ncand(fc);
        float jp[3];
        rows_of(fc, pc, al, jp);
FB_UNROLL
        for (int k = 0; k < 3; k++) fb_st_scr(pc + (NC_JP + k)*BLK, jp[k]);
      }
    }
    *g0_out = g0; *pp_out = pp;
  }

  /* ---- sweep C (first Newton iteration only): leaves -> root, M p from the rigid bodies'
   * forces, written where the next sweep A expects the previous gradient; returns p'Mp.  The
   * first step is the large one (|p| ~ 60 |a|): taking M(a1 - a0) = alpha M p from the bodies
   * instead of from H p = -g makes the second iteration refine its rounding error. */
  FB_MEM float newton_c() {
    const int nb = m.nbody;
    float fc6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float pMp = 0.f;
    float nx[7];      /* pure acceleration[6], p of the next body to visit */
    const int n_it = SPLIT ? ord_n : nb - 1;
    {
      const float *pn = nblock(SPLIT ? (ord_n > 0 ? ord[ord_n - 1] : 1) : nb - 1);
FB_UNROLL
      for (int k = 0; k < 6; k++) nx[k] = fb_ld_scr(pn + (NB_AP + k)*BLK);
      nx[6] = fb_ld_scr(pn + NB_P*BLK);
    }
    for (int i = n_it; i >= 0; i--) {
      if (SPLIT && i == ord_bnd) this->split_barrier();
      if (i == 0) break;
      const int b = SPLIT ? ord[i - 1] : i;
      const int bn = SPLIT ? (i >= 2 ? ord[i - 2] : 0) : (i > 1 ? i - 1 : 0);
      const FastRec &rc = rec[b];
      FB_PIN_I(rc.jtype); FB_PIN_I(rc.flags); FB_PIN_I(rc.pblk); FB_PIN_I(rc.parent);
      FB_PIN_F(rc.mass); FB_PIN_F(rc.armature);
FB_UNROLL
      for (int k = 0; k < 3; k++) { FB_PIN_F(rc.hloc[k]); FB_PIN_F(rc.axis[k]); }
FB_UNROLL
      for (int k = 0; k < 5; k++) FB_PIN_F(rc.Ib[k]);
      const float *pb = block(b);
      float *pn = nblock(b);
      const int jtype = rc.jtype, flags = rc.flags;
      float al[6];
FB_UNROLL
      for (int k = 0; k < 6; k++) al[k] = nx[k];
      const float pj = nx[6];
      if (bn) {
        const float *pn1 = nblock(bn);
FB_UNROLL
        for (int k = 0; k < 6; k++) nx[k] = fb_ld_scr(pn1 + (NB_AP + k)*BLK);
        nx[6] = fb_ld_scr(pn1 + NB_P*BLK);
      }
      float R[9], h[3], Iw[6], F[6];
      body_frame(rc, pb, R, h, Iw);
      {
        /* f = m (a_lin + alpha x h),  n = Iw alpha + h x f */
        float cr[3], t[3];
        v_cross(al, h, cr);
FB_UNROLL
        for (int k = 0; k < 3; k++) F[3 + k] = rc.mass*(al[3 + k] + cr[k]);
        sym_mul(Iw, al, t);
        v_cross(h, F + 3, cr);
FB_UNROLL
        for (int k = 0; k < 3; k++) F[k] = t[k] + cr[k];
      }
      if (flags & FT_ADD_CARRY) {
FB_UNROLL
        for (int k = 0; k < 6; k++) F[k] += fc6[k];
      }
      if (flags & FT_HAS_SLOT) {
        const float *so = slot(rc.slot);
FB_UNROLL
        for (int k = 0; k < 6; k++) F[k] += so[(21 + k)*BLK];
      }
      if (jtype == FB_JNT_FREE) {
        float *pr = nroot();
FB_UNROLL
        for (int k = 0; k < 6; k++) {
          fb_st_scr(pr + (NR_MD + k)*BLK, F[k]);
          pMp += F[k]*fb_ld_scr(pr + (NR_P + k)*BLK);
        }
        continue;
      }
      if (jtype >= 0) {
        float ax[3];
        m_rot(R, rc.axis[0], rc.axis[1], rc.axis[2], ax);
        const float mp = ((LEAN || jtype == FB_JNT_HINGE) ? ax[0]*F[0] + ax[1]*F[1] + ax[2]*F[2]
                                                : ax[0]*F[3] + ax[1]*F[4] + ax[2]*F[5]) + rc.armature*pj;
        fb_st_scr(pn + NB_MD*BLK, mp);
        pMp += pj*mp;
      }
      if (rc.parent == 0) continue;
      {
        const float *pp = (s + rc.pblk*BLK);
        float r[3], cr[3];
FB_UNROLL
        for (int k = 0; k < 3; k++) r[k] = pb[(FB_ORG + k)*BLK] - pp[(FB_ORG + k)*BLK];
        v_cross(r, F + 3, cr);
        F[0] += cr[0]; F[1] += cr[1]; F[2] += cr[2];
      }
      if (flags & FT_TO_CARRY) {
FB_UNROLL
        for (int k = 0; k < 6; k++) fc6[k] = F[k];
      } else {
        float *so = slot(rc.pslot);
        if (flags & FT_FIRST_WRITER) {
FB_UNROLL
          for (int k = 0; k < 6; k++) so[(21 + k)*BLK] = F[k];
        } else {
FB_UNROLL
          for (int k = 0; k < 6; k++) so[(21 + k)*BLK] += F[k];
        }
      }
    }
    return pMp;
  }

  /* Row sums of the line search at N step lengths a[i] in one pass over the rows some lane holds
   * active: S = sum_active D jp (res + a jp), Q = sum_active D jp^2, and a hash of the active set.
   * The loads of a row block are issued one visit ahead. */
  template <int N>
  FB_MEM void line_eval(const float *a, float *S, float *Q, unsigned *hash) const {
FB_UNROLL
    for (int i = 0; i < N; i++) { S[i] = 0.f; Q[i] = 0.f; hash[i] = 0u; }
FB_UNROLL
    for (int w = 0; w < 2; w++) {
      for (unsigned mw = lany[w]; mw; mw &= mw - 1) {
        const int b = 32*w + FB_FFS(mw) - 1;
        const float *pn = nblock(b);
        const float dlo = fb_ld_scr(pn + NB_DLO*BLK), dhi = fb_ld_scr(pn + NB_DHI*BLK);
        const float arlo = fb_ld_scr(pn + NB_ARLO*BLK), arhi = fb_ld_scr(pn + NB_ARHI*BLK);
        const float aj = fb_ld_scr(pn + NB_A*BLK), pj = fb_ld_scr(pn + NB_P*BLK);
FB_UNROLL
        for (int i = 0; i < N; i++) {
          const float xl = (aj - arlo) + a[i]*pj, xh = (-aj - arhi) - a[i]*pj;
          const int al_ = dlo > 0.f && xl < 0.f, ah_ = dhi > 0.f && xh < 0.f;
          if (al_) { S[i] += dlo*pj*xl; Q[i] += dlo*pj*pj; }
          if (ah_) { S[i] -= dhi*pj*xh; Q[i] += dhi*pj*pj; }
          hash[i] = (hash[i] + (unsigned)(al_ + 2*ah_))*0x9E3779B1u;
        }
      }
    }
    CandIter it = cand_begin();
    int fc = cand_next(it);
    float nx[7];
    if (fc >= 0) {
      const float *pc = ncand(fc);
FB_UNROLL
      for (int k = 0; k < 7; k++) nx[k] = fb_ld_scr(pc + (NC_D + k)*BLK);     /* D, res[3], jp[3] are contiguous */
    }
    while (fc >= 0) {
      const float D = lane_on(fc) ? nx[0] : 0.f;
      const float rn = nx[1], r1 = nx[2], r2 = nx[3], jn = nx[4], j1 = nx[5], j2 = nx[6];
      fc = cand_next(it);
      if (fc >= 0) {
        const float *pc = ncand(fc);
FB_UNROLL
        for (int k = 0; k < 7; k++) nx[k] = fb_ld_scr(pc + (NC_D + k)*BLK);
      }
FB_UNROLL
      for (int row = 0; row < 4; row++) {
        const float sg = (row & 1) ? -1.f : 1.f;
        const float res = rn + sg*(row < 2 ? r1 : r2), jp = jn + sg*(row < 2 ? j1 : j2);
        const float djp = D*jp;
FB_UNROLL
        for (int i = 0; i < N; i++) {
          const float x = res + a[i]*jp;
          const int act = D > 0.f && x < 0.f;
          if (act) { S[i] += djp*x; Q[i] += djp*jp; }
          hash[i] = (hash[i] + (unsigned)act)*0x9E3779B1u;
        }
      }
    }
  }

  /* a <- a + alpha p for everything that is carried, and the forces of the rows that switched,
   * Delta = D res' ([was active] - [is active]), for the next sweep A.  mode 1: before the first
   * iteration -- nothing moves, nothing was active (Delta = the constraint forces at a0).  mode 2:
   * after the first iteration -- the next gradient starts from M(a1 - a0) (sweep C), so Delta is
   * the whole constraint force at a1.  Returns |a|^2. */
  FB_MEM float newton_update(float alpha, int mode) {
    const int nb = m.nbody;
    const int first = mode == 1, fresh = mode != 0;
    float a2 = 0.f;
    /* four joints per round: their loads are in flight together */
    for (int b0 = 1; b0 < nb; b0 += 4) {
      float av[4], pv[4];
FB_UNROLL
      for (int i = 0; i < 4; i++) {
        const int b = b0 + i;
        av[i] = 0.f; pv[i] = 0.f;
        if (b < nb && owns(b)) {
          const float *pn = nblock(b);
          av[i] = fb_ld_scr(pn + NB_A*BLK);
          if (!first) pv[i] = fb_ld_scr(pn + NB_P*BLK);
        }
      }
FB_UNROLL
      for (int i = 0; i < 4; i++) {
        const int b = b0 + i;
        if (b >= nb || !owns(b)) continue;
        const FastRec &rc = rec[b];
        float *pn = nblock(b);
        if (rc.jtype == FB_JNT_FREE) {
          if (first) continue;
          float *pr = nroot();
          float ra[6], rp[6];
FB_UNROLL
          for (int k = 0; k < 6; k++) { ra[k] = fb_ld_scr(pr + (NR_A + k)*BLK); rp[k] = fb_ld_scr(pr + (NR_P + k)*BLK); }
FB_UNROLL
          for (int k = 0; k < 6; k++) {
            const float an = ra[k] + alpha*rp[k];
            fb_st_scr(pr + (NR_A + k)*BLK, an);
            a2 += an*an;
          }
        } else if (rc.jtype >= 0) {
          const float ao = av[i];
          const float an = first ? ao : ao + alpha*pv[i];
          if (!first) fb_st_scr(pn + NB_A*BLK, an);
          a2 += an*an;
          if ((rc.flags & FT_LIMITED) && lim_on(b)) {
            const float dlo = fb_ld_scr(pn + NB_DLO*BLK), dhi = fb_ld_scr(pn + NB_DHI*BLK);
            const float arlo = fb_ld_scr(pn + NB_ARLO*BLK), arhi = fb_ld_scr(pn + NB_ARHI*BLK);
            const float rlo = an - arlo, rhi = -an - arhi;
            const int wl = !fresh && dlo > 0.f && ao - arlo < 0.f, il = dlo > 0.f && rlo < 0.f;
            const int wh = !fresh && dhi > 0.f && -ao - arhi < 0.f, ih = dhi > 0.f && rhi < 0.f;
            /* row Jacobians +1 / -1 */
            fb_st_scr(pn + NB_MP*BLK, dlo*rlo*(float)(wl - il) - dhi*rhi*(float)(wh - ih));
          }
        }
      }
    }
    CandIter it = cand_begin();
    for (int fc = cand_next(it); fc >= 0; fc = cand_next(it)) {
      float *pc = ncand(fc);
      const float mu = cand_mu(crec[fc]);
      float v[7];
FB_UNROLL
      for (int k = 0; k < 7; k++) v[k] = fb_ld_scr(pc + (NC_D + k)*BLK);     /* D, res[3], jp[3] */
      const float D = lane_on(fc) ? v[0] : 0.f;
      float rn[3];
FB_UNROLL
      for (int k = 0; k < 3; k++) rn[k] = first ? v[1 + k] : v[1 + k] + alpha*v[4 + k];
      float d4[4];
FB_UNROLL
      for (int row = 0; row < 4; row++) {
        const float sg = (row & 1) ? -1.f : 1.f;
        const float ro = v[1] + sg*(row < 2 ? v[2] : v[3]), rw = rn[0] + sg*(row < 2 ? rn[1] : rn[2]);
        const int was = !fresh && D > 0.f && ro < 0.f, is = D > 0.f && rw < 0.f;
        d4[row] = D*rw*(float)(was - is);
      }
      if (!first) {
FB_UNROLL
        for (int k = 0; k < 3; k++) fb_st_scr(pc + (NC_RES + k)*BLK, rn[k]);
      }
      fb_st_scr(pc + NC_JP*BLK, d4[0] + d4[1] + d4[2] + d4[3]);
      fb_st_scr(pc + (NC_JP + 1)*BLK, mu*(d4[0] - d4[1]));
      fb_st_scr(pc + (NC_JP + 2)*BLK, mu*(d4[2] - d4[3]));
    }
    return a2;
  }

  /* ---- primal Newton with exact line search (SURVEY.md A.8), matrix-free */
  FB_MEM void solve(int mine) {      /* SPLIT: `mine` as combined over the warps */
    int done = !mine;
    const int maxit = m.solver_iterations < 50 ? m.solver_iterations : 50;
    int it = 0;
    float prev_ratio = 3.0e38f, keep = 1.f;
    newton_update(0.f, 1);      /* Delta = the constraint forces at a0: g = -J' f(a0) */
    for (; it < maxit && FB_ANY(!done); it++) {
      float pg, pp, gv, sl;
      unsigned hash, hash0;
      newton_a(keep);
      newton_b(&pg, &pp, it == 0);
      /* Line search on phi'(a) = p'M(a - a0) + a p'Mp + sum_active(a) D jp (res + a jp).  With
       * H p = -g:  p'M(a - a0) = p.g - S(0),  p'Mp = -p.g - Q(0).  First iteration: a = a0 and
       * p'Mp comes from sweep C.  phi'(0) = p.g and phi''(0) = -p.g, so the first trial step is
       * the full Newton step: the rows are evaluated at 0 and 1 in the same pass. */
      const float a01[2] = {0.f, 1.f};
      float S2[2], Q2[2];
      unsigned h2[2];
      line_eval<2>(a01, S2, Q2, h2);
      if (SPLIT) {
        float f6[6] = {pg, pp, S2[0], S2[1], Q2[0], Q2[1]};
        h2[0] *= hmul; h2[1] *= hmul;
        rcombine<6, 2>(f6, h2);
        pg = f6[0]; pp = f6[1]; S2[0] = f6[2]; S2[1] = f6[3]; Q2[0] = f6[4]; Q2[1] = f6[5];
      }
      float g0 = pg - S2[0], pMp = fmaxf(-pg - Q2[0], 1e-7f*fabsf(pg));
      if (it == 0) {
        g0 = 0.f; pMp = newton_c();
        if (SPLIT) rcombine<1, 0>(&pMp, 0);
      }
      /* zero of the piecewise-linear derivative by safeguarded Newton steps */
      int ls_done = done || !(pg < 0.f), nls = 1, exact = 0;
      float a = ls_done ? 0.f : 1.f, lo = 0.f, hi = 3.0e38f;
      gv = g0 + pMp + S2[1]; sl = pMp + Q2[1];
      hash0 = h2[0]; hash = h2[1];
      for (int ls = 1; ls < 16 && FB_ANY(!ls_done); ls++) {
        /* here gv, sl, hash belong to a */
        if (!ls_done) {
          if (fabsf(gv) <= 1e-5f*fabsf(pg)) {
            /* The derivative vanishes at a with the rows that were active at 0: H was built from
             * the final active set, the Newton step is the exact minimiser, nothing is left to do. */
            exact = hash == hash0;
            ls_done = 1;
          } else {
            if (gv < 0.f) lo = a; else hi = a;
            float an = a - gv/sl;
            if (!(an > lo) || !(an < hi)) {
              if (hi < 1.0e38f) an = 0.5f*(lo + hi);
              else an = 2.f*a + 1.f;
            }
            /* the derivative is piecewise linear: a Newton step inside one piece is exact, and the
             * outer iteration absorbs what is left (MuJoCo's own search stops at 1e-2) */
            if (fabsf(an - a) <= 1e-4f*fabsf(an)) ls_done = 1;
            a = an;
          }
        }
        if (!FB_ANY(!ls_done)) break;
        nls++;
        float S1, Q1;
        line_eval<1>(&a, &S1, &Q1, &hash);
        if (SPLIT) {
          float f2[2] = {S1, Q1};
          hash *= hmul;
          rcombine<2, 1>(f2, &hash);
          S1 = f2[0]; Q1 = f2[1];
        }
        gv = g0 + a*pMp + S1; sl = pMp + Q1;
      }
      if (done) a = 0.f;
      float a2 = newton_update(a, it == 0 ? 2 : 0);
      if (SPLIT) rcombine<1, 0>(&a2, 0);
      keep = it == 0 ? a : 1.f - a;
      /* Stop on a relative step below 3e-5 (|alpha p|^2 <= 1e-9 |a|^2).  Convergence is quadratic
       * once the active set is right -- measured relative steps 6e1, 4e-1, 1e-2, then the fp32
       * floor of 1e-6 .. 4e-6 -- so the step after a 1e-2 one is already rounding noise; MuJoCo's
       * own tests (scaled gradient / improvement below 1e-8) are out of reach of fp32.  Also stop
       * when the step has stopped shrinking below 1e-3: that is the floor of a worse-conditioned
       * model. */
      const float ratio = a*a*pp, lim = 1e-9f*a2 + 1e-30f;
      if (!done && (exact || ratio <= lim || (it > 0 && ratio <= 1e-6f*a2 && ratio >= 0.25f*prev_ratio))) done = 1;
      /* a diverged environment (non-finite state) must not hold its warp in the loop */
      if (!(a2 < 3.0e38f) || !(ratio < 3.0e38f)) done = 1;
      prev_ratio = ratio;
#ifdef FB_HOST_EMU
      if (fb_emu_stats && role == 0) { fb_emu_stats[0] += 1; fb_emu_stats[1] += nls; }
#endif
    }
#ifdef FB_HOST_EMU
    if (fb_emu_stats && role == 0) fb_emu_stats[2] += 1;
#endif
    if (!done) FB_FLAG_OR(P.flags + env, FB_FLAG_SOLVER);
  }

  /* ---- constraint forces of the solution: limit torques and sensor values per joint, world
   * force / contact-frame force / world position per candidate */
  FB_MEM void final_forces() {
    const int nb = m.nbody;
    for (int b = 1; b < nb; b++) {
      const FastRec &rc = rec[b];
      if (!owns(b) || rc.jtype < 0 || rc.jtype == FB_JNT_FREE) continue;
      float *pn = nblock(b);
      float tauc = 0.f, lf = 0.f;
      if ((rc.flags & FT_LIMITED) && lim_on(b)) {
        const float dlo = fb_ld_scr(pn + NB_DLO*BLK), dhi = fb_ld_scr(pn + NB_DHI*BLK);
        const float aj = fb_ld_scr(pn + NB_A*BLK);
        const float rlo = aj - fb_ld_scr(pn + NB_ARLO*BLK), rhi = -aj - fb_ld_scr(pn + NB_ARHI*BLK);
        const float flo = (dlo > 0.f && rlo < 0.f) ? -dlo*rlo : 0.f;
        const float fhi = (dhi > 0.f && rhi < 0.f) ? -dhi*rhi : 0.f;
        tauc = flo - fhi;
        /* jointlimitfrc: efc_force of the joint's first active limit row */
        lf = dlo > 0.f ? flo : (dhi > 0.f ? fhi : 0.f);
      }
      fb_st_scr(pn + NB_TAUC*BLK, tauc);
      fb_st_scr(pn + NB_LIMF*BLK, lf);
    }
    CandIter it = cand_begin();
    for (int fc = cand_next(it); fc >= 0; fc = cand_next(it)) {
      const CandRec &cr_ = crec[fc];
      float *pc = ncand(fc);
      const float *pb = s + cr_.pblk*BLK;
      const float D = lane_on(fc) ? fb_ld_scr(pc + NC_D*BLK) : 0.f;
      float n[3] = {cr_.pn[0], cr_.pn[1], cr_.pn[2]}, t1[3], t2[3];
FB_UNROLL
      for (int k = 0; k < 3; k++) t1[k] = fb_ld_scr(pc + (NC_T1 + k)*BLK);
      v_cross(n, t1, t2);
      const float mu = cand_mu(cr_);
      const float rn = fb_ld_scr(pc + NC_RES*BLK), r1 = fb_ld_scr(pc + (NC_RES + 1)*BLK), r2 = fb_ld_scr(pc + (NC_RES + 2)*BLK);
      float f4[4];
FB_UNROLL
      for (int row = 0; row < 4; row++) {
        const float res = rn + ((row & 1) ? -1.f : 1.f)*(row < 2 ? r1 : r2);
        f4[row] = (D > 0.f && res < 0.f) ? -D*res : 0.f;
      }
      const float fn = f4[0] + f4[1] + f4[2] + f4[3], ft1 = mu*(f4[0] - f4[1]), ft2 = mu*(f4[2] - f4[3]);
      fb_st_scr(pc + NC_JP*BLK, fn); fb_st_scr(pc + (NC_JP + 1)*BLK, ft1); fb_st_scr(pc + (NC_JP + 2)*BLK, ft2);
FB_UNROLL
      for (int k = 0; k < 3; k++) {
        fb_st_scr(pc + (NC_RES + k)*BLK, fn*n[k] + ft1*t1[k] + ft2*t2[k]);
        fb_st_scr(pc + (NC_POS + k)*BLK, rootpos[k] + pb[(FB_ORG + k)*BLK] + fb_ld_scr(pc + (NC_R + k)*BLK));
      }
    }
  }

  /* ---- contacts rows: sensors.pyx:140-190 over the active candidates */
  FB_MEM void write_contacts(float *row_contacts) {
    const long long ev = P.env_pad*FB_VEC_CONTACTS;
    /* SPLIT: a sensor may sum candidates of several warps' bodies.  The masks are disjoint over the
     * warps: their sums are the masks of the whole tree (and the barrier of the reduction makes the
     * other warps' forces visible); the sensors are then dealt over the warps. */
    unsigned long long keep_m[4] = {hm[0], hm[1], hany[0], hany[1]};
    if (SPLIT) {
      unsigned u8[8];
FB_UNROLL
      for (int k = 0; k < 4; k++) { u8[2*k] = (unsigned)keep_m[k]; u8[2*k + 1] = (unsigned)(keep_m[k] >> 32); }
      rcombine<0, 8>(0, u8);
      hm[0] = u8[0] | ((unsigned long long)u8[1] << 32); hm[1] = u8[2] | ((unsigned long long)u8[3] << 32);
      hany[0] = u8[4] | ((unsigned long long)u8[5] << 32); hany[1] = u8[6] | ((unsigned long long)u8[7] << 32);
    }
    for (int sx = SPLIT ? role : 0; sx < m.n_contacts; sx += SPLIT ? nroles : 1) {
      float acc[12], nsum = 0.f;
FB_UNROLL
      for (int k = 0; k < 12; k++) acc[k] = 0.f;
      for (int t = MI(ft_sstart, sx); t < MI(ft_sstart, sx + 1); t++) {
        const int fc = MI(ft_scand, t);
        if (!any_on(fc)) continue;
        const CandRec &cr_ = crec[fc];
        const float *pc = ncand(fc);
        const float sg = lane_on(fc) ? MF(ft_ssign, t) : 0.f;
        float n[3] = {cr_.pn[0], cr_.pn[1], cr_.pn[2]}, t1[3], t2[3], tot[3];
FB_UNROLL
        for (int k = 0; k < 3; k++) t1[k] = fb_ld_scr(pc + (NC_T1 + k)*BLK);
        v_cross(n, t1, t2);
        const float fn = fb_ld_scr(pc + NC_JP*BLK), f1 = fb_ld_scr(pc + (NC_JP + 1)*BLK), f2 = fb_ld_scr(pc + (NC_JP + 2)*BLK);
        if (sg == 0.f) continue;
FB_UNROLL
        for (int k = 0; k < 3; k++) {
          const float re = sg*fn*n[k], fri = sg*f1*t1[k] + sg*f2*t2[k];
          acc[k] += re; acc[3 + k] += fri; tot[k] = re + fri; acc[6 + k] += tot[k];
        }
        const float nrm = sqrtf(tot[0]*tot[0] + tot[1]*tot[1] + tot[2]*tot[2]);
FB_UNROLL
        for (int k = 0; k < 3; k++) acc[9 + k] += nrm*fb_ld_scr(pc + (NC_POS + k)*BLK);
        nsum += nrm;
      }
      const float ip = (nsum > 0.f ? 1.0f/nsum : 1.0f)*m.inv_meters, in = m.inv_newtons;
      float *row = row_contacts + (long long)(3*sx)*ev;
      fb_st4(row, acc[0]*in, acc[1]*in, acc[2]*in, acc[3]*in);
      fb_st4(row + ev, acc[4]*in, acc[5]*in, acc[6]*in, acc[7]*in);
      fb_st4(row + 2*ev, acc[8]*in, acc[9]*ip, acc[10]*ip, acc[11]*ip);
    }
    if (SPLIT) { hm[0] = keep_m[0]; hm[1] = keep_m[1]; hany[0] = keep_m[2]; hany[1] = keep_m[3]; }
  }

  /* Steps k0 .. n_steps-1 of the launch, constraints included. */
  FB_MEM void run_con(int k0, int coop, int lane) {
    this->load_state(coop, lane);
    const size_t e = (size_t)env;
    const int n = P.n_steps;
    long long row = (P.it0 + k0) % P.ring;
    for (int k = k0; k < n; k++) {
      row = row + 1 == P.ring ? 0 : row + 1;
      float *row_links = fb_log_row(P.log_links, row, m.n_links*20, P.env_pad, FB_VEC_LINKS, e);
      float *row_joints = fb_log_row(P.log_joints, row, m.n_joints*m.joint_cols, P.env_pad, FB_VEC_JOINTS, e);
      float *row_contacts = fb_log_row(P.log_contacts, row, m.n_contacts*12, P.env_pad, FB_VEC_CONTACTS, e);
      float *row_xfrc = fb_log_row(P.log_xfrc, row, m.n_xfrc*6, P.env_pad, FB_VEC_XFRC, e);
      const float time = (float)this->episode_it(P.it0 + k)*m.timestep;
      const int maybe = this->pass_poses(row_links);
      if (rec[1].jtype == FB_JNT_FREE) { rt[3] = rqn[0]; rt[4] = rqn[1]; rt[5] = rqn[2]; rt[6] = rqn[3]; }
      float aroot[6] = {0.f, 0.f, 0.f, -m.grav[0], -m.grav[1], -m.grav[2]};
      const float *seqk = P.ctrl_seq ? P.ctrl_seq + ((size_t)(P.seq_pos + k)*P.seq_stride)*P.env_pad + e : 0;
      const int store_ctrl = k == n - 1 && m.n_wc > 0;
      int mine = 0, bad;
      if (FB_ANY(maybe)) mine = detect();
      this->zfill = this->log_row_dirty(P.it0 + k + 1);
      if (FB_ANY(mine)) {
        this->dirty_c = P.it0 + k + 1;       /* every lane of the warp writes the constraint columns of this row */
        this->template pass_inertia_m<1>(time, aroot, 0, seqk);
        smooth_accel(aroot);
        solve(mine);
        final_forces();
FB_UNROLL
        for (int i = 0; i < 3; i++) { aroot[i] = 0.f; aroot[3 + i] = -m.grav[i]; }
        this->template pass_inertia_m<2>(time, aroot, store_ctrl, seqk);
        bad = this->template pass_accel_m<1>(aroot, row_joints, row_xfrc);
        write_contacts(row_contacts);
      } else {
        this->template pass_inertia_m<0>(time, aroot, store_ctrl, seqk);
        bad = this->template pass_accel_m<0>(aroot, row_joints, row_xfrc);
        if (this->zfill) this->zero_contacts(row_contacts);
      }
      if (bad) FB_FLAG_OR(P.flags + env, FB_FLAG_NONFINITE);
    }
    if (P.ctrl_seq) this->store_seq_end(n);
    P.con_dirty[env] = this->dirty_c;
    this->store_state(P.it0 + n, coop, lane);
  }

  /* SPLIT: run_con from step 0 for a block whose warps step the SAME environments, each its own
   * bodies (split_setup + con_split_setup).  Warp 0 owns the root state and the state I/O; every
   * thread of the block takes every barrier. */
  FB_MEM void run_con_split(int coop, int lane) {
    if (role == 0) this->load_state(coop, lane);
    FB_BLOCK_BARRIER();
    const size_t e = (size_t)env;
    const int n = P.n_steps;
    long long row = P.it0 % P.ring;
    idle = 0;
    for (int k = 0; k < n; k++) {
      row = row + 1 == P.ring ? 0 : row + 1;
      float *row_links = fb_log_row(P.log_links, row, m.n_links*20, P.env_pad, FB_VEC_LINKS, e);
      float *row_joints = fb_log_row(P.log_joints, row, m.n_joints*m.joint_cols, P.env_pad, FB_VEC_JOINTS, e);
      float *row_contacts = fb_log_row(P.log_contacts, row, m.n_contacts*12, P.env_pad, FB_VEC_CONTACTS, e);
      float *row_xfrc = fb_log_row(P.log_xfrc, row, m.n_xfrc*6, P.env_pad, FB_VEC_XFRC, e);
      const float time = (float)this->episode_it(P.it0 + k)*m.timestep;
      const int maybe = rany(this->pass_poses(row_links));
      if (role == 0 && rec[1].jtype == FB_JNT_FREE) { rt[3] = rqn[0]; rt[4] = rqn[1]; rt[5] = rqn[2]; rt[6] = rqn[3]; }
      float aroot[6] = {0.f, 0.f, 0.f, -m.grav[0], -m.grav[1], -m.grav[2]};
      const float *seqk = P.ctrl_seq ? P.ctrl_seq + ((size_t)(P.seq_pos + k)*P.seq_stride)*P.env_pad + e : 0;
      const int store_ctrl = k == n - 1 && m.n_wc > 0;
      int mine = 0, bad;
      if (FB_ANY(maybe)) mine = rany(detect());
      this->zfill = this->log_row_dirty(P.it0 + k + 1);
      if (FB_ANY(mine)) {
        this->dirty_c = P.it0 + k + 1;
        this->template pass_inertia_m<1>(time, aroot, 0, seqk);
        FB_BLOCK_BARRIER();
        smooth_accel(aroot);
        solve(mine);
        final_forces();
FB_UNROLL
        for (int i = 0; i < 3; i++) { aroot[i] = 0.f; aroot[3 + i] = -m.grav[i]; }
        FB_BLOCK_BARRIER();
        this->template pass_inertia_m<2>(time, aroot, store_ctrl, seqk);
        FB_BLOCK_BARRIER();
        bad = this->template pass_accel_m<1>(aroot, row_joints, row_xfrc);
        write_contacts(row_contacts);
      } else {
        this->template pass_inertia_m<0>(time, aroot, store_ctrl, seqk);
        FB_BLOCK_BARRIER();
        bad = this->template pass_accel_m<0>(aroot, row_joints, row_xfrc);
        if (this->zfill && role == 0) this->zero_contacts(row_contacts);
      }
      if (bad) FB_FLAG_OR(P.flags + env, FB_FLAG_NONFINITE);
      FB_BLOCK_BARRIER();
    }
    if (role != 0) return;
    if (P.ctrl_seq) this->store_seq_end(n);
    P.con_dirty[env] = this->dirty_c;
    this->store_state(P.it0 + n, coop, lane);
  }
};

#endif /* FB_FASTC_H_ */
