/*
 * fb_fast.h -- the environment-per-thread step: ONE CUDA thread advances one
 * environment while no joint limit or contact is active.
 *
 * Every environment runs the same model, so a warp of 32 environments executes
 * the same tree walk with the same (uniform) indices: no divergence, no
 * shuffles, no barriers, every lane busy.  Forward dynamics is the
 * articulated-body recursion (three sweeps over the bodies), which needs no
 * mass matrix and therefore a per-environment working set small enough to keep
 * 64 environments per SM resident in shared memory.  Implicit joint damping of
 * the Euler integrator, (M + h D) x = f (SURVEY.md A.10), is the same recursion
 * with h*damping added to the joint-space diagonal, so the result is the x the
 * team path (fb_device.h: CRB + L'DL, as MuJoCo does it) computes, up to fp32
 * rounding.
 *
 * Spatial vectors are [angular; linear] in WORLD axes, taken about the body's
 * own reference point (its joint anchor); moving a quantity from a body to its
 * parent is a pure translation by r = anchor(body) - anchor(parent), built from
 * the parent rotation and model constants (never from differences of world
 * positions), which keeps every number at link scale in fp32.
 *
 * As soon as pass 1 of a step sees a joint limit violated or a body inside the
 * conservative contact bound of a plane, the environment stops here with its
 * state untouched and is appended to the pending list; the team kernel
 * (fb_device.h) takes it over from that step with the full constraint solver.
 *
 * Shared-memory layout: element i of a per-environment array lives at
 * (off + i)*BLK + thread (DevFastLayout), i.e. consecutive lanes hit consecutive
 * banks.
 *
 * Reference anchors: step order mj_step via farms_mujoco/simulation/
 * simulation.py:156; log rows farms_mujoco/simulation/physics.py:435-524;
 * drag/buoyancy farms_mujoco/swimming/drag.pyx:152-268,389-411; hook order
 * farms_mujoco/simulation/task.py:168-186.
 */
#ifndef FB_FAST_H_
#define FB_FAST_H_

#include "fb_device.h"

#ifdef FB_HOST_EMU
FB_DEV void fb_st4(float *p, float a, float b, float c, float d) { p[0] = a; p[1] = b; p[2] = c; p[3] = d; }
FB_DEV void fb_st2(float *p, float a, float b) { p[0] = a; p[1] = b; }
#else
/* log rows are written once and not read back by the step: streaming (evict-first) stores
 * keep them from pushing the L2-resident scratch out */
FB_DEV void fb_st4(float *p, float a, float b, float c, float d) {
  __stcs(reinterpret_cast<float4 *>(p), make_float4(a, b, c, d));
}
FB_DEV void fb_st2(float *p, float a, float b) { __stcs(reinterpret_cast<float2 *>(p), make_float2(a, b)); }
#endif

/* bit i (0..127) of a two-word mask held in registers */
FB_DEV int fb_bit128(const unsigned long long *m2, int i) {
  return (int)(((i < 64 ? m2[0] : m2[1]) >> (i & 63)) & 1ull);
}

/* articulated inertia about a point, world axes:  [ A  H ] [w]   A, M symmetric
 *                                                 [ H' M ] [v]   (xx yy zz xy xz yz) */
struct ArtInertia {
  float A[6], H[9], M[6];
};

FB_DEV void sym_mul(const float *S, const float *x, float *y) {
  y[0] = S[0]*x[0] + S[3]*x[1] + S[4]*x[2];
  y[1] = S[3]*x[0] + S[1]*x[1] + S[5]*x[2];
  y[2] = S[4]*x[0] + S[5]*x[1] + S[2]*x[2];
}
/* y = H x, y = H' x */
FB_DEV void h_mul(const float *H, const float *x, float *y) {
  y[0] = H[0]*x[0] + H[1]*x[1] + H[2]*x[2];
  y[1] = H[3]*x[0] + H[4]*x[1] + H[5]*x[2];
  y[2] = H[6]*x[0] + H[7]*x[1] + H[8]*x[2];
}
FB_DEV void ht_mul(const float *H, const float *x, float *y) {
  y[0] = H[0]*x[0] + H[3]*x[1] + H[6]*x[2];
  y[1] = H[1]*x[0] + H[4]*x[1] + H[7]*x[2];
  y[2] = H[2]*x[0] + H[5]*x[1] + H[8]*x[2];
}
/* S -= k * a a' (symmetric rank one) */
FB_DEV void sym_rank1(float *S, const float *a, float k) {
  float b0 = k*a[0], b1 = k*a[1], b2 = k*a[2];
  S[0] -= b0*a[0]; S[1] -= b1*a[1]; S[2] -= b2*a[2];
  S[3] -= b0*a[1]; S[4] -= b0*a[2]; S[5] -= b1*a[2];
}

/* Move an articulated inertia and a force from a point to the point -r away
 * (child anchor -> parent anchor, r = child - parent):
 *   H' = H + r~ M,  A' = A - H r~ + r~ H''  ,  n' = n + r x f          */
FB_DEV void art_shift(ArtInertia &I, float *p, const float *r) {
  float Mc[3][3] = {{I.M[0], I.M[3], I.M[4]}, {I.M[3], I.M[1], I.M[5]}, {I.M[4], I.M[5], I.M[2]}};
  float Hn[9];
FB_UNROLL
  for (int j = 0; j < 3; j++) {
    float c[3];
    v_cross(r, Mc[j], c);                       /* column j of r~ M */
    Hn[j] = I.H[j] + c[0]; Hn[3 + j] = I.H[3 + j] + c[1]; Hn[6 + j] = I.H[6 + j] + c[2];
  }
  float T[9];                                   /* T = -H r~ + r~ Hn' */
FB_UNROLL
  for (int i = 0; i < 3; i++) {
    float hr[3];
    v_cross(I.H + 3*i, r, hr);                  /* row i of H r~ */
    T[3*i] = -hr[0]; T[3*i+1] = -hr[1]; T[3*i+2] = -hr[2];
  }
FB_UNROLL
  for (int j = 0; j < 3; j++) {
    float rh[3];
    v_cross(r, Hn + 3*j, rh);                   /* column j of r~ Hn' */
    T[j] += rh[0]; T[3 + j] += rh[1]; T[6 + j] += rh[2];
  }
  I.A[0] += T[0]; I.A[1] += T[4]; I.A[2] += T[8];
  I.A[3] += 0.5f*(T[1] + T[3]); I.A[4] += 0.5f*(T[2] + T[6]); I.A[5] += 0.5f*(T[5] + T[7]);
FB_UNROLL
  for (int k = 0; k < 9; k++) I.H[k] = Hn[k];
  float c[3];
  v_cross(r, p + 3, c);
  p[0] += c[0]; p[1] += c[1]; p[2] += c[2];
}

/* solve the symmetric positive definite 6x6 system K x = b in registers (L D L') */
FB_DEV void solve6(float K[6][6], const float *b, float *x) {
  float dinv[6];
FB_UNROLL
  for (int j = 0; j < 6; j++) {
    float d = K[j][j];
FB_UNROLL
    for (int k = 0; k < j; k++) d -= K[j][k]*K[j][k]*K[k][k];
    K[j][j] = d;
    dinv[j] = 1.0f/d;
FB_UNROLL
    for (int i = j + 1; i < 6; i++) {
      float v = K[i][j];
FB_UNROLL
      for (int k = 0; k < j; k++) v -= K[i][k]*K[j][k]*K[k][k];
      K[i][j] = v*dinv[j];
    }
  }
  float y[6];
FB_UNROLL
  for (int i = 0; i < 6; i++) {
    float v = b[i];
FB_UNROLL
    for (int k = 0; k < i; k++) v -= K[i][k]*y[k];
    y[i] = v;
  }
FB_UNROLL
  for (int i = 5; i >= 0; i--) {
    float v = y[i]*dinv[i];
FB_UNROLL
    for (int k = i + 1; k < 6; k++) v -= K[k][i]*x[k];
    x[i] = v;
  }
}

#ifdef FB_HOST_EMU
FB_DEV float fb_rcp(float x) { return 1.0f/x; }
FB_DEV float fb_ld_scr(const float *p) { return *p; }
FB_DEV void fb_st_scr(float *p, float v) { *p = v; }
#else
FB_DEV float fb_rcp(float x) { return __frcp_rn(x); }
/* the scratch lives in L2: bypass L1 both ways */
FB_DEV float fb_ld_scr(const float *p) { return __ldcg(p); }
FB_DEV void fb_st_scr(float *p, float v) { __stcg(p, v); }
#endif

/* sin and cos of a half joint angle: minimax polynomials on |x| <= pi/4 (the cephes sinf /
 * cosf kernels, < 1 ulp), the library sincosf beyond (|joint angle| > pi/2 is rare) */
FB_DEV void fb_sincos_half(float x, float *sn, float *cs) {
  if (fabsf(x) <= 0.78539816f) {
    const float z = x*x;
    *sn = x + x*z*(-1.6666654611e-1f + z*(8.3321608736e-3f + z*(-1.9515295891e-4f)));
    *cs = 1.0f - 0.5f*z + z*z*(4.166664568298827e-2f + z*(-1.388731625493765e-3f + z*2.443315711809948e-5f));
  } else {
    fb_sincos(x, sn, cs);
  }
}

/* Pin a constant-bank value into a register at this point of the program: ptxas otherwise
 * issues the indexed LDC right before the first use and the lone warp of the scheduler waits
 * out its latency every time. */
#ifdef FB_HOST_EMU
#define FB_PIN_F(x) (void)(x)
#define FB_PIN_I(x) (void)(x)
#define FB_ANY(p) (p)
#else
/* warp vote at a point every live lane of the warp reaches together */
#define FB_ANY(p) __any_sync(__activemask(), (p))
#define FB_PIN_F(x) asm volatile("" :: "f"(x))
#define FB_PIN_I(x) asm volatile("" :: "r"(x))
#endif

template <int SYNC> FB_DEV void fb_block_sync() {
#ifndef FB_HOST_EMU
  if (SYNC) __syncthreads();
#endif
}

/* SLIM = 1 (large batches, unconstrained kernel only): the shared-memory block of a body holds
 * its pose only (7 floats); velocities and the accumulation slots of the branching bodies move to
 * the L2 scratch, fetched one body ahead like the rest of it.  203 instead of 431 floats of
 * shared memory per SALAMANDER: 8 warps of environments per SM instead of 4, i.e. two warps per
 * scheduler to hide each other's latencies, which pays once the batch has that many warps. */
/* LEAN = 1: the model (DevFastLayout::lean) has hinge joints only, anchors at the body origins,
 * axisymmetric inertias, the linear actuation form on every joint and the farms joints-row layout,
 * and the launch reads no control sequence: the slide-joint, general-inertia, generic-actuation,
 * anchor-offset and generic-column paths are compiled out.  Same arithmetic on the paths that
 * remain (bit-identical results); the point is the SIZE of the three body loops -- they run out of
 * a 32 KB instruction cache, and unrolling them by two (60 KB) was measured 10-25 % slower. */
/* SPLIT = 1 (small batches, regular layout): the 32 environments of a block are stepped by several
 * warps, each visiting its own bodies of the tree in two phases per sweep (FastSplit, fb_model.h);
 * the per-body code is the one every other variant runs, in the same order along every chain, so
 * the results are bit-identical to the single-warp kernel. */
/* ENVP = 1 (fb_set_env_param): joint stiffness and damping, drag coefficients, water velocity,
 * actuator gains and biases come from the per-environment tables (FbEnvTables, `ept`) where one is
 * set (a uniform null test per table), else from the records / the model as with ENVP = 0; the
 * records' linear actuation form (Kq, Kqd, T0 and the unlogged KqU, KqdU, T0U) from the table the
 * host derives from the biases (FbEnvTables::lin).  Same arithmetic on the values. */
/* the tables' pointer is a member of the ENVP variants only: a member that the other variants never
 * read still changed how ptxas scheduled the SLIM kernels.  The ENVP variants also run the episode
 * clock (fb_reset_envs): the wave controller's time is formed from episode_it(it0 + k), with the
 * environment's episode start loaded once per launch (0 while FbEnvTables::episode_start is not
 * bound, which gives the same value as it0 + k). */
template <int ENVP> struct FbEnvRef {
  const FbEnvTables *ept;   /* the per-environment parameter tables (kernel parameters) */
  long long ep0;            /* batch iteration of this environment's episode row 0 */
  FB_MEM FbEnvRef(const FbEnvTables *ept_, int env) : ept(ept_), ep0(ept_->episode_start ? ept_->episode_start[env] : 0) {}
  FB_MEM long long episode_it(long long it) const { return it - ep0; }
};
template <> struct FbEnvRef<0> {
  FB_MEM FbEnvRef(const FbEnvTables *, int) {}
  FB_MEM long long episode_it(long long it) const { return it; }
};
template <int BLK, int SLIM = 0, int LEAN = 0, int SPLIT = 0, int ENVP = 0> struct FbFast : FbEnvRef<ENVP> {
  /* SLIM scratch block: W[6] U 1/d trq q qd V[6] tc tu -- the first 17 are one contiguous run */
  enum { NF = SLIM ? 7 : FB_NF, GNF = SLIM ? FG_NF + 6 : FG_NF, FG_V = SLIM ? 11 : FG_NF,
         FGTC = SLIM ? 17 : FG_TC, FGTU = SLIM ? 18 : FG_TU };
  const FbParams &P;
  const DevModel &m;
  const FastRec *rec; /* [nbody], constant bank (kernel parameters) */
  float *s;           /* shared floats, already offset by the thread index */
  const int env;
  float *gs;          /* global scratch of this thread: element i at gs[i*BLK] ([warp][field][lane]) */
  float env_phase;
  float rt[13];       /* floating root: qpos[7], qvel[6] (registers) */
  float rootpos[3];   /* world position the anchors are measured from (the floating root) */
  float rqn[4];       /* normalised root quaternion of the current step */
  /* constrained step (fb_fastc.h; unused on the unconstrained kernel): scratch like gs, the
   * candidate records, and the masks of the candidates that touch in this lane / in any lane */
  float *cs, *csc;
  const CandRec *crec;
  unsigned long long hm[2], hany[2];
  /* log columns only a constrained step can make non-zero (contacts rows, joint_limit_force) are
   * zero-filled by an unconstrained step only when the ring row it overwrites may hold such a
   * value: dirty_c = last iteration a constraint-capable kernel wrote a row of this environment
   * (FbParams::con_dirty), zfill = verdict for the current step */
  long long dirty_c;
  int zfill;
  /* SPLIT: this warp's body list (ascending; phase A = [0, ord_bnd)), its role (0 = the trunk warp,
   * which also owns the root state and the state I/O), whether this lane's environment has left
   * the kernel (it still takes every barrier), the root position as warp 0 publishes it and the
   * per-lane hand-over flags the warps agree through */
  const uint8_t *ord;
  int ord_n, ord_bnd, role, idle;
  float *sroot;
  int *sflag;

  FB_MEM FbFast(const FbParams &P_, const FastRec *rec_, float *s_, float *gs_, int env_, const FbEnvTables *ept_ = 0)
      : FbEnvRef<ENVP>(ept_, env_), P(P_), m(P_.m), rec(rec_), s(s_), env(env_), gs(gs_), cs(0), csc(0), crec(0) {
    env_phase = P.env_phase[env];
    dirty_c = P.con_dirty[env];
    zfill = 1;
    ord = 0; ord_n = 0; ord_bnd = 0; role = 0; idle = 0; sroot = 0; sflag = 0;
    rootpos[0] = rootpos[1] = rootpos[2] = 0.f;
    rqn[0] = 1.f; rqn[1] = rqn[2] = rqn[3] = 0.f;
FB_UNROLL
    for (int k = 0; k < 13; k++) rt[k] = 0.f;
  }

  FB_MEM void split_setup(const FastSplit &sp, int role_, float *sroot_, int *sflag_) {
    role = role_; ord = sp.order[role_]; ord_n = sp.n[role_]; ord_bnd = sp.boundary[role_];
    sroot = sroot_; sflag = sflag_;
  }
  /* phase barrier of a sweep (every thread of the block, idle or not) */
  FB_MEM void split_barrier() const { FB_BLOCK_BARRIER(); }
  /* row of iteration `itr` (before the ring modulus): was it last written at or before dirty_c? */
  FB_MEM int log_row_dirty(long long itr) const {
    const long long prev = itr - P.ring;
    return prev >= 0 && prev <= dirty_c;
  }
  FB_MEM float *block(int b) const { return s + (m.X.body0 + NF*(b - 1))*BLK; }
  FB_MEM float *gblock(int b) const { return gs + GNF*(b - 1)*BLK; }
  /* accumulation slot i: shared memory, or (SLIM) the scratch behind the body blocks */
  FB_MEM float *slot(int i) const {
    return SLIM ? gs + (GNF*(m.nbody - 1) + 27*i)*BLK : s + (m.X.slots + 27*i)*BLK;
  }
  FB_MEM float sl_ld(const float *so, int k) const { return SLIM ? fb_ld_scr(so + k*BLK) : so[k*BLK]; }
  FB_MEM void sl_st(float *so, int k, float v) const { if (SLIM) fb_st_scr(so + k*BLK, v); else so[k*BLK] = v; }
  FB_MEM void sl_add(float *so, int k, float v) const { sl_st(so, k, sl_ld(so, k) + v); }
  /* shared-memory block of the parent */
  FB_MEM const float *pblock(const FastRec &rc) const { return s + (SLIM ? rc.pblk7 : rc.pblk)*BLK; }
  FB_MEM float *nblock(int b) const { return cs + NB_NF*(b - 1)*BLK; }
  FB_MEM float *nroot() const { return cs + NB_NF*(m.nbody - 1)*BLK; }
  FB_MEM float *ncand(int fc) const { return csc + NC_NF*BLK*fc; }

  /* actuator a's gain, entry i of the biases ([nu][3]) and term k of the joint's linear actuation
   * form (FbEnvTables::lin; `model`: the record's value): this environment's where ENVP and a table */
  FB_MEM float gain_of(int a) const {
    if constexpr (ENVP != 0) if (this->ept->gain) return this->ept->gain[(size_t)a*P.env_pad + env];
    return MF(act_gain, a);
  }
  FB_MEM float bias_of(int i) const {
    if constexpr (ENVP != 0) if (this->ept->bias) return this->ept->bias[(size_t)i*P.env_pad + env];
    return MF(act_bias, i);
  }
  FB_MEM float lin_of(const FastRec &rc, int k, float model) const {
    if constexpr (ENVP != 0) if (this->ept->lin) return this->ept->lin[(size_t)(6*rc.jid + k)*P.env_pad + env];
    return model;
  }

  /* generic actuation (clamps, gears, partial logging): force sum and farms joint_torque */
  /* ctrl of actuator a at this step: the uploaded sequence when there is one, else the held value */
  FB_MEM float ctrl_of(int a, const float *seqk) const {
    return seqk ? seqk[(long long)a*P.env_pad] : P.ctrl[(size_t)env*m.nu + a];
  }

  /* per-step constants of a joint's linear actuation form (load_state does this once when ctrl is held) */
  FB_MEM void seq_constants(const FastRec &rc, const float *seqk, float *tc, float *tu) const {
    float c = lin_of(rc, 2, rc.T0), u = lin_of(rc, 5, rc.T0U);
    int ap = -1, av = -1, at = -1;
    if (rc.fj >= 0) { ap = MI(fj_actpos, rc.fj); av = MI(fj_actvel, rc.fj); at = MI(fj_acttrq, rc.fj); }
    for (int t = MI(jnt_actstart, rc.jid); t < MI(jnt_actstart, rc.jid + 1); t++) {
      int a = MI(act_sorted, t);
      if (a == rc.wave_act || MI(ft_actoff, a)) continue;
      float f = gain_of(a)*seqk[(long long)a*P.env_pad];
      c += f;
      if (!(a == ap || a == av || a == at)) u += f;
    }
    *tc = c; *tu = u;
  }

  FB_MEM void actuation_generic(const FastRec &rc, float q, float qd, float time, int store_ctrl,
                                const float *seqk, float *tau, float *trq_log) const {
    const int jid = rc.jid, fj = rc.fj;
    int a0 = MI(jnt_actstart, jid), a1 = MI(jnt_actstart, jid + 1);
    int ap = -1, av = -1, at = -1;
    if (fj >= 0) { ap = MI(fj_actpos, fj); av = MI(fj_actvel, fj); at = MI(fj_acttrq, fj); }
    float tsum = 0.f, lsum = 0.f;
    for (int t = a0; t < a1; t++) {
      int a = MI(act_sorted, t);
      float gear = MF(act_gear, a);
      int w = MI(ft_actwc, a);
      float c;
      if (w >= 0) {
        float ph = 6.283185307179586f*MF(wc_freq, w)*time - MF(wc_lag, w) + env_phase;
        c = MF(wc_off, w) + MF(wc_amp, w)*sinf(ph);
        if (store_ctrl) P.ctrl[(size_t)env*m.nu + a] = c;
      } else {
        c = ctrl_of(a, seqk);
      }
      if (MI(act_ctrllimited, a)) c = fminf(MF(act_ctrlrange, 2*a+1), fmaxf(MF(act_ctrlrange, 2*a), c));
      float f = gain_of(a)*c + bias_of(3*a) + bias_of(3*a+1)*(gear*q) + bias_of(3*a+2)*(gear*qd);
      if (MI(act_forcelimited, a)) f = fminf(MF(act_forcerange, 2*a+1), fmaxf(MF(act_forcerange, 2*a), f));
      tsum += gear*f;
      if (a == ap || a == av || a == at) lsum += f;
    }
    *tau = tsum;
    *trq_log = lsum;
  }

  /* qpos_spring ends a launch as the last sequence entry used, as if the host had set it step by
   * step (task.py:338-346); `last` = that step's rows of this environment */
  FB_MEM void store_springrefs(const float *last) const {
    if (P.n_spring <= 0) return;
    for (int b = 1; b < m.nbody; b++)
      if (FT_SREF(rec[b].flags) >= 0) P.qpos_spring[(size_t)env*m.nq + rec[b].qa] = last[(long long)(m.nu + FT_SREF(rec[b].flags))*P.env_pad];
  }
  /* end of a launch of n steps with a control sequence: ctrl ends as the last entry used, as if
   * the host had set it step by step (the wave-driven actuators keep what the last step wrote) */
  FB_MEM void store_seq_end(int n) const {
    const size_t e = (size_t)env;
    const float *last = P.ctrl_seq + ((size_t)(P.seq_pos + n - 1)*P.seq_stride)*P.env_pad + e;
    for (int a = 0; a < m.nu; a++)
      if (MI(ft_actwc, a) < 0) P.ctrl[e*m.nu + a] = last[(long long)a*P.env_pad];
    store_springrefs(last);
  }
  /* no contact is active in this step: its contacts row is zero (sensors.pyx:140-190) */
  FB_MEM void zero_contacts(float *row_contacts) const {
    for (int i = 0; i < m.n_contacts*3; i++) fb_st4(row_contacts + i*(P.env_pad*FB_VEC_CONTACTS), 0.f, 0.f, 0.f, 0.f);
  }

  /* joint half of load_state: root state into registers, q / qd and the constant part of the
   * actuation of every joint into the scratch */
  FB_MEM void load_joints(const float *gq, const float *gv, const float *g_ctrl) {
    for (int b = 1; b < m.nbody; b++) {
      const FastRec &rc = rec[b];
      float *pg = gblock(b);
      if (rc.jtype == FB_JNT_FREE) {
FB_UNROLL
        for (int k = 0; k < 7; k++) rt[k] = gq[rc.qa + k];
FB_UNROLL
        for (int k = 0; k < 6; k++) rt[7 + k] = gv[rc.da + k];
      } else if (rc.jtype >= 0) {
        fb_st_scr(pg + FG_Q*BLK, gq[rc.qa]);
        fb_st_scr(pg + FG_QD*BLK, gv[rc.da]);
        /* constant part of the joint's actuation over this launch (ctrl is held), and of
         * the actuators the farms joint_torque column leaves out */
        float tc = lin_of(rc, 2, rc.T0), tu = lin_of(rc, 5, rc.T0U);
        if (rc.flags & FT_ACT_SIMPLE) {
          int ap = -1, av = -1, at = -1;
          if (rc.fj >= 0) { ap = MI(fj_actpos, rc.fj); av = MI(fj_actvel, rc.fj); at = MI(fj_acttrq, rc.fj); }
          for (int t = MI(jnt_actstart, rc.jid); t < MI(jnt_actstart, rc.jid + 1); t++) {
            int a = MI(act_sorted, t);
            if (a == rc.wave_act || MI(ft_actoff, a)) continue;
            float f = gain_of(a)*g_ctrl[a];
            tc += f;
            if (!(a == ap || a == av || a == at)) tu += f;
          }
        }
        fb_st_scr(pg + FGTC*BLK, tc);
        fb_st_scr(pg + FGTU*BLK, tu);
      }
    }
  }
  FB_MEM void load_wrenches(const float *gx) {
    for (int b = 1; b < m.nbody; b++) {
      float *pg = gblock(b);
      for (int k = 0; k < 6; k++) fb_st_scr(pg + (FG_W + k)*BLK, gx[6*b + k]);
    }
  }

  /* State enters and leaves through a shared-memory tile when the warp is full: the
   * warp copies the contiguous [32 envs][n] blocks of qpos / qvel / ctrl / xfrc_applied with
   * coalesced accesses and every thread then picks its own row from the tile (the body blocks
   * are not live outside the step loop).  coop = 1: one tile holds everything; coop = 2 (SLIM
   * layout, smaller blocks): joints first, wrenches second; coop = 0: plain per-thread accesses. */
  FB_MEM void load_state(int coop, int lane) {
    const int nq = m.nq, nv = m.nv, nu = m.nu > 0 ? m.nu : 1, nx = 6*m.nbody;
    const float *gq = P.qpos + (size_t)env*nq, *gv = P.qvel + (size_t)env*nv;
    const float *gx = P.xfrc_applied + (size_t)env*nx;
    const float *g_ctrl = P.ctrl + (size_t)env*nu;
#ifndef FB_HOST_EMU
    if (coop) {
      float *tile = s - lane;
      const size_t e0 = (size_t)(env - lane);
      for (int i = lane; i < 32*nq; i += 32) tile[i] = P.qpos[e0*nq + i];
      for (int i = lane; i < 32*nv; i += 32) tile[32*nq + i] = P.qvel[e0*nv + i];
      for (int i = lane; i < 32*nu; i += 32) tile[32*(nq + nv) + i] = P.ctrl[e0*nu + i];
      if (coop == 1) for (int i = lane; i < 32*nx; i += 32) tile[32*(nq + nv + nu) + i] = P.xfrc_applied[e0*nx + i];
      __syncwarp();
      gq = tile + lane*nq; gv = tile + 32*nq + lane*nv;
      g_ctrl = tile + 32*(nq + nv) + lane*nu; gx = tile + 32*(nq + nv + nu) + lane*nx;
      if (coop == 2) {
        load_joints(gq, gv, g_ctrl);
        __syncwarp();
        for (int i = lane; i < 32*nx; i += 32) tile[i] = P.xfrc_applied[e0*nx + i];
        __syncwarp();
        load_wrenches(tile + lane*nx);
        __syncwarp();
        return;
      }
    }
#endif
    load_joints(gq, gv, g_ctrl);
    load_wrenches(gx);
#ifndef FB_HOST_EMU
    if (coop) __syncwarp();      /* the tile becomes the body blocks */
#endif
  }

  FB_MEM void store_joints(float *gq, float *gv) const {
    for (int b = 1; b < m.nbody; b++) {
      const FastRec &rc = rec[b];
      const float *pg = gblock(b);
      if (rc.jtype == FB_JNT_FREE) {
FB_UNROLL
        for (int k = 0; k < 7; k++) gq[rc.qa + k] = rt[k];
FB_UNROLL
        for (int k = 0; k < 6; k++) gv[rc.da + k] = rt[7 + k];
      } else if (rc.jtype >= 0) {
        gq[rc.qa] = fb_ld_scr(pg + FG_Q*BLK);
        gv[rc.da] = fb_ld_scr(pg + FG_QD*BLK);
      }
    }
  }
  FB_MEM void store_wrenches(float *gx) const {
    for (int b = 1; b < m.nbody; b++) {
      const float *pg = gblock(b);
      for (int k = 0; k < 6; k++) gx[6*b + k] = fb_ld_scr(pg + (FG_W + k)*BLK);
    }
  }

  FB_MEM void store_state(long long iteration, int coop, int lane) {
    const int nq = m.nq, nv = m.nv, nx = 6*m.nbody;
    float *gq = P.qpos + (size_t)env*nq, *gv = P.qvel + (size_t)env*nv;
    float *gx = P.xfrc_applied + (size_t)env*nx;
#ifndef FB_HOST_EMU
    if (coop == 2) {
      __syncwarp();              /* every lane is done with its body blocks */
      float *tile = s - lane;
      const size_t e0 = (size_t)(env - lane);
      store_joints(tile + lane*nq, tile + 32*nq + lane*nv);
      __syncwarp();
      for (int i = lane; i < 32*nq; i += 32) P.qpos[e0*nq + i] = tile[i];
      for (int i = lane; i < 32*nv; i += 32) P.qvel[e0*nv + i] = tile[32*nq + i];
      __syncwarp();
      gx = tile + lane*nx;
      for (int k = 0; k < 6; k++) gx[k] = 0.f;      /* the world body carries no wrench */
      store_wrenches(gx);
      __syncwarp();
      for (int i = lane; i < 32*nx; i += 32) P.xfrc_applied[e0*nx + i] = tile[i];
      P.iteration[env] = iteration;
      return;
    }
    if (coop) {
      __syncwarp();              /* every lane is done with its body blocks */
      float *tile = s - lane;
      gq = tile + lane*nq; gv = tile + 32*nq + lane*nv; gx = tile + 32*(nq + nv) + lane*nx;
      for (int k = 0; k < 6; k++) gx[k] = 0.f;      /* the world body carries no wrench */
    }
#endif
    store_joints(gq, gv);
    store_wrenches(gx);
#ifndef FB_HOST_EMU
    if (coop) {
      __syncwarp();
      const float *tile = s - lane;
      const size_t e0 = (size_t)(env - lane);
      for (int i = lane; i < 32*nq; i += 32) P.qpos[e0*nq + i] = tile[i];
      for (int i = lane; i < 32*nv; i += 32) P.qvel[e0*nv + i] = tile[32*nq + i];
      for (int i = lane; i < 32*nx; i += 32) P.xfrc_applied[e0*nx + i] = tile[32*(nq + nv) + i];
    }
#endif
    P.iteration[env] = iteration;
  }

  /* ---- pass 1: poses, velocities, links rows, constraint detection.  Returns 1
   * when a limit or a plane bound is active (the step must not be taken here). */
  FB_MEM int pass_poses(float *row_links) {
    const int nb = m.nbody;
    int active = 0;
    /* scratch values are fetched one body ahead: the L2 round trip overlaps the arithmetic */
    const int b0 = SPLIT ? (ord_n > 0 ? ord[0] : 1) : 1;
    float nq = fb_ld_scr(gblock(b0) + FG_Q*BLK), nqd = fb_ld_scr(gblock(b0) + FG_QD*BLK);
    const int n_it = SPLIT ? ord_n : nb - 1;
    float *pb = block(1) - NF*BLK;
    float *pn = gblock(1);
    Quat lastq = {1.f, 0.f, 0.f, 0.f};
    float lasto[3] = {0.f, 0.f, 0.f}, lastv[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float lastR[9] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f};
    /* SLIM: velocity of the parent of a branch child (its parent is not the previous body), fetched
     * from the scratch while the previous body is computed -- issued at its use it cost a full L2
     * round trip per branch (r1aq: 6 % of the stall samples together with its pass-3 twin) */
    float nvp[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int i = 0; i <= n_it; i++) {
      if (SPLIT && i == ord_bnd) {
        split_barrier();                 /* the trunk is placed: the subtrees hanging off it start */
        if (role != 0 && rec[1].jtype == FB_JNT_FREE) {       /* (a fixed base: the anchors are measured from the world origin) */
FB_UNROLL
          for (int k = 0; k < 3; k++) rootpos[k] = sroot[k*BLK];
        }
      }
      if (i == n_it) break;
      if (SPLIT && idle) continue;
      const int b = SPLIT ? ord[i] : i + 1;
      const int bn = SPLIT ? (i + 1 < n_it ? ord[i + 1] : 0) : (i + 2 < nb ? i + 2 : 0);   /* visited next; 0: none */
      const FastRec &rc0 = rec[b];
      struct { int parent, jtype, flags, pblk, link, chk0, chk1; float dpos[3], bquat[4], axis[3], qpos0, lo, hi, margin, hloc[3], chk[4], jpos[3]; } rc;
      rc.parent = rc0.parent; rc.jtype = rc0.jtype; rc.flags = rc0.flags; rc.pblk = SLIM ? rc0.pblk7 : rc0.pblk; rc.link = rc0.link;
      rc.chk0 = rc0.chk0; rc.chk1 = rc0.chk1; rc.qpos0 = rc0.qpos0; rc.lo = rc0.lo; rc.hi = rc0.hi; rc.margin = rc0.margin;
FB_UNROLL
      for (int k = 0; k < 3; k++) { rc.dpos[k] = rc0.dpos[k]; rc.axis[k] = rc0.axis[k]; rc.hloc[k] = rc0.hloc[k]; rc.jpos[k] = rc0.jpos[k]; }
FB_UNROLL
      for (int k = 0; k < 4; k++) { rc.bquat[k] = rc0.bquat[k]; rc.chk[k] = rc0.chk[k]; }
      FB_PIN_I(rc.parent); FB_PIN_I(rc.jtype); FB_PIN_I(rc.flags); FB_PIN_I(rc.pblk); FB_PIN_I(rc.link);
      FB_PIN_F(rc.qpos0); FB_PIN_F(rc.lo); FB_PIN_F(rc.hi); FB_PIN_F(rc.margin);
FB_UNROLL
      for (int k = 0; k < 3; k++) { FB_PIN_F(rc.dpos[k]); FB_PIN_F(rc.axis[k]); FB_PIN_F(rc.hloc[k]); }
FB_UNROLL
      for (int k = 0; k < 4; k++) { FB_PIN_F(rc.bquat[k]); FB_PIN_F(rc.chk[k]); }
      if (SPLIT) { pb = block(b); pn = gblock(bn ? bn : b); }
      else { pb += NF*BLK; pn += GNF*BLK; }
      const float cq = nq, cqd = nqd;
      if (bn) { nq = fb_ld_scr(pn + FG_Q*BLK); nqd = fb_ld_scr(pn + FG_QD*BLK); }
      float *pgv = SPLIT ? gblock(b) : pn - GNF*BLK;       /* scratch block of this body (pn runs one ahead) */
      const int jtype = rc.jtype;
      Quat q;
      float o[3], v[6], R[9];
      /* pose / velocity / rotation of body b-1, still in registers for a chain child */
      const Quat ql_ = lastq;
      float lo_[3], lv_[6], lR_[9];
FB_UNROLL
      for (int k = 0; k < 3; k++) lo_[k] = lasto[k];
FB_UNROLL
      for (int k = 0; k < 6; k++) lv_[k] = lastv[k];
FB_UNROLL
      for (int k = 0; k < 9; k++) lR_[k] = lastR[k];
      if (jtype == FB_JNT_FREE) {
        Quat qq = {rt[3], rt[4], rt[5], rt[6]};
        q = q_normalize(qq);
        /* qpos takes the normalised quaternion (mj_kinematics does it in place) only once the
         * step is known to be taken here: a handed-over environment must reach the team kernel
         * with its state bit-for-bit untouched */
        rqn[0] = q.w; rqn[1] = q.x; rqn[2] = q.y; rqn[3] = q.z;
        q_mat(q, R);
FB_UNROLL
        for (int k = 0; k < 3; k++) { rootpos[k] = rt[k]; o[k] = 0.f; v[3 + k] = rt[7 + k]; }
        if (SPLIT) {
FB_UNROLL
          for (int k = 0; k < 3; k++) sroot[k*BLK] = rt[k];
        }
        m_rot(R, rt[10], rt[11], rt[12], v);
      } else {
        Quat qp = {1.f, 0.f, 0.f, 0.f};
        float op[3] = {0.f, 0.f, 0.f}, vp[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        float Rp[9], r[3], dq = 0.f, qd = 0.f;
        if (rc.flags & FT_TO_CARRY) {
          /* the parent is the previous body: its pose is still in registers */
          qp = ql_;
FB_UNROLL
          for (int k = 0; k < 3; k++) op[k] = lo_[k];
FB_UNROLL
          for (int k = 0; k < 6; k++) vp[k] = lv_[k];
FB_UNROLL
          for (int k = 0; k < 9; k++) Rp[k] = lR_[k];
        } else {
          if (rc.parent > 0) {
            const float *pp = (s + rc.pblk*BLK);
            qp.w = pp[(FB_QUAT)*BLK]; qp.x = pp[(FB_QUAT + 1)*BLK]; qp.y = pp[(FB_QUAT + 2)*BLK]; qp.z = pp[(FB_QUAT + 3)*BLK];
FB_UNROLL
            for (int k = 0; k < 3; k++) op[k] = pp[(FB_ORG + k)*BLK];
            if (SLIM) {
FB_UNROLL
              for (int k = 0; k < 6; k++) vp[k] = nvp[k];
            } else {
FB_UNROLL
              for (int k = 0; k < 6; k++) vp[k] = pp[(FB_VEL + k)*BLK];
            }
          }
          q_mat(qp, Rp);
        }
        m_rot(Rp, rc.dpos[0], rc.dpos[1], rc.dpos[2], r);
        Quat bq = {rc.bquat[0], rc.bquat[1], rc.bquat[2], rc.bquat[3]};
        q = q_mul(qp, bq);
        if (!LEAN && (rc.flags & FT_HAS_JPOS)) {      /* the anchor is fixed in the frame before the joint rotation */
          float Rpre[9], t[3];
          q_mat(q_normalize(q), Rpre);
          m_rot(Rpre, rc.jpos[0], rc.jpos[1], rc.jpos[2], t);
          r[0] += t[0]; r[1] += t[1]; r[2] += t[2];
        }
        if (jtype >= 0) {
          const float qj = cq;
          qd = cqd;
          dq = qj - rc.qpos0;
          if (LEAN || jtype == FB_JNT_HINGE) {
            float sn, cs;
            fb_sincos_half(0.5f*dq, &sn, &cs);
            Quat ql = {cs, rc.axis[0]*sn, rc.axis[1]*sn, rc.axis[2]*sn};
            q = q_mul(q, ql);
          }
          if ((rc.flags & FT_LIMITED) && (qj - rc.lo < rc.margin || rc.hi - qj < rc.margin)) active = 1;
        }
        q = q_normalize(q);
        q_mat(q, R);
        float ax[3] = {0.f, 0.f, 0.f}, cr[3];
        if (jtype >= 0) m_rot(R, rc.axis[0], rc.axis[1], rc.axis[2], ax);
        if (!LEAN && jtype == FB_JNT_SLIDE) { r[0] += ax[0]*dq; r[1] += ax[1]*dq; r[2] += ax[2]*dq; }
        v_cross(vp, r, cr);                      /* w_parent x r */
FB_UNROLL
        for (int k = 0; k < 3; k++) {
          o[k] = op[k] + r[k];
          v[k] = vp[k] + (jtype == FB_JNT_HINGE ? ax[k]*qd : 0.f);
          v[3 + k] = vp[3 + k] + cr[k] + (!LEAN && jtype == FB_JNT_SLIDE ? ax[k]*qd : 0.f);
        }
      }
      if (SLIM && b + 1 < nb) {
        const FastRec &rn = rec[b + 1];
        if (!(rn.flags & FT_TO_CARRY) && rn.parent > 0) {      /* parent <= b - 1: its velocity is stored */
          const float *pgp = gs + GNF*(rn.parent - 1)*BLK;
FB_UNROLL
          for (int k = 0; k < 6; k++) nvp[k] = fb_ld_scr(pgp + (FG_V + k)*BLK);
        }
      }
      pb[(FB_QUAT)*BLK] = q.w; pb[(FB_QUAT + 1)*BLK] = q.x; pb[(FB_QUAT + 2)*BLK] = q.y; pb[(FB_QUAT + 3)*BLK] = q.z;
FB_UNROLL
      for (int k = 0; k < 3; k++) pb[(FB_ORG + k)*BLK] = o[k];
      if (SLIM) {
FB_UNROLL
        for (int k = 0; k < 6; k++) fb_st_scr(pgv + (FG_V + k)*BLK, v[k]);
      } else {
FB_UNROLL
        for (int k = 0; k < 6; k++) pb[(FB_VEL + k)*BLK] = v[k];
      }
      lastq = q;
FB_UNROLL
      for (int k = 0; k < 3; k++) lasto[k] = o[k];
FB_UNROLL
      for (int k = 0; k < 6; k++) lastv[k] = v[k];
FB_UNROLL
      for (int k = 0; k < 9; k++) lastR[k] = R[k];
      float xpos[3] = {rootpos[0] + o[0], rootpos[1] + o[1], rootpos[2] + o[2]};
      if (!LEAN && (rc.flags & FT_HAS_JPOS)) {
        float t[3];
        m_rot(R, rc.jpos[0], rc.jpos[1], rc.jpos[2], t);
        xpos[0] -= t[0]; xpos[1] -= t[1]; xpos[2] -= t[2];
      }
      /* conservative plane bound */
      if (rc.chk[0]*xpos[0] + rc.chk[1]*xpos[1] + rc.chk[2]*xpos[2] < rc.chk[3]) active = 1;
      for (int t = rc.chk0; t < rc.chk1; t++)
        if (MF(ft_chk, 4*t)*xpos[0] + MF(ft_chk, 4*t+1)*xpos[1] + MF(ft_chk, 4*t+2)*xpos[2] < MF(ft_chk, 4*t+3)) active = 1;
      /* links row: physics.py:449-466 + :435-446 */
      if (rc.link >= 0) {
        float h[3], cr[3];
        m_rot(R, rc.hloc[0], rc.hloc[1], rc.hloc[2], h);   /* com - anchor */
        v_cross(v, h, cr);
        const float im = m.inv_meters, iv = m.inv_velocity, iw = m.inv_angvel;
        const long long ev = P.env_pad*FB_VEC_LINKS;
        float *row = row_links + (long long)(5*rc.link)*ev;     /* five 16-byte vectors, each coalesced across the warp */
        fb_st4(row, (rootpos[0] + o[0] + h[0])*im, (rootpos[1] + o[1] + h[1])*im, (rootpos[2] + o[2] + h[2])*im, q.x);
        fb_st4(row + ev, q.y, q.z, q.w, xpos[0]*im);
        fb_st4(row + 2*ev, xpos[1]*im, xpos[2]*im, q.x, q.y);
        fb_st4(row + 3*ev, q.z, q.w, (v[3] + cr[0])*iv, (v[4] + cr[1])*iv);
        fb_st4(row + 4*ev, (v[5] + cr[2])*iv, v[0]*iw, v[1]*iw, v[2]*iw);
      }
    }
    return active;
  }

  /* ---- pass 2: leaves -> root, articulated inertias and bias forces.
   * MODE 0: the step, (M + h D) x = f.  MODE 1 (constrained step): M a0 = f, the unconstrained
   * acceleration; U, u, 1/d go to the constraint scratch and the applied wrench stays where it is.
   * MODE 2 (constrained step): MODE 0 with the constraint forces applied (contact forces as body
   * wrenches, limit forces as joint torques). */
  FB_MEM void pass_inertia(float time, float *aroot, int store_ctrl, const float *seqk) {
    pass_inertia_m<0>(time, aroot, store_ctrl, seqk);
  }
  template <int MODE>
  FB_MEM void pass_inertia_m(float time, float *aroot, int store_ctrl, const float *seqk) {
    const int nb = m.nbody;
    const float hdt = m.timestep;
    ArtInertia C;        /* carry from child b+1 */
    float pc[6];
FB_UNROLL
    for (int k = 0; k < 6; k++) { C.A[k] = 0.f; C.M[k] = 0.f; pc[k] = 0.f; }
FB_UNROLL
    for (int k = 0; k < 9; k++) C.H[k] = 0.f;
    float nx[10] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};        /* W[6], q, qd, tc, tu of the next body to visit */
    float nxv[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};     /* SLIM: its velocity */
    const int n_it = SPLIT ? ord_n : nb - 1;
    {
      const float *pn = gblock(SPLIT ? (ord_n > 0 ? ord[ord_n - 1] : 1) : nb - 1);
FB_UNROLL
      for (int k = 0; k < 6; k++) nx[k] = fb_ld_scr(pn + (FG_W + k)*BLK);
      nx[6] = fb_ld_scr(pn + FG_Q*BLK); nx[7] = fb_ld_scr(pn + FG_QD*BLK);
      nx[8] = fb_ld_scr(pn + FGTC*BLK); nx[9] = fb_ld_scr(pn + FGTU*BLK);
      if (SLIM) {
FB_UNROLL
        for (int k = 0; k < 6; k++) nxv[k] = fb_ld_scr(pn + (FG_V + k)*BLK);
      }
    }
    float *pb = block(nb - 1) + NF*BLK;
    float *pg = gblock(nb - 1) + GNF*BLK;
    for (int i = n_it; i >= 0; i--) {
      if (SPLIT && i == ord_bnd) split_barrier();      /* the subtrees have handed over: the trunk goes on */
      if (i == 0) break;
      if (SPLIT && idle) continue;
      const int b = SPLIT ? ord[i - 1] : i;
      const int bn = SPLIT ? (i >= 2 ? ord[i - 2] : 0) : (i > 1 ? i - 1 : 0);
      const FastRec &rc = rec[b];
      /* issue the record loads of this body now (see FB_PIN_F) */
      FB_PIN_I(rc.jtype); FB_PIN_I(rc.flags); FB_PIN_I(SLIM ? rc.pblk7 : rc.pblk); FB_PIN_I(rc.parent);
      FB_PIN_F(rc.mass); FB_PIN_F(rc.Kq); FB_PIN_F(rc.Kqd); FB_PIN_F(rc.KqU); FB_PIN_F(rc.KqdU);
      FB_PIN_F(rc.wfreq); FB_PIN_F(rc.wlag); FB_PIN_F(rc.woff); FB_PIN_F(rc.wamp); FB_PIN_F(rc.wgain);
      FB_PIN_F(rc.stiffness); FB_PIN_F(rc.damping); FB_PIN_F(rc.armature);
FB_UNROLL
      for (int k = 0; k < 3; k++) { FB_PIN_F(rc.hloc[k]); FB_PIN_F(rc.axis[k]); }
FB_UNROLL
      for (int k = 0; k < 5; k++) FB_PIN_F(rc.Ib[k]);
      /* ENVP: this environment's values, loads issued here */
      float estiff = 0.f, edamp = 0.f, eKq = 0.f, eKqd = 0.f, eKqU = 0.f, eKqdU = 0.f, ewgain = 0.f;
      if constexpr (ENVP) {
        const FbEnvTables *ept = this->ept;
        estiff = rc.stiffness; edamp = rc.damping;
        eKq = rc.Kq; eKqd = rc.Kqd; eKqU = rc.KqU; eKqdU = rc.KqdU; ewgain = rc.wgain;
        if (rc.jtype > FB_JNT_FREE) {
          if (ept->stiffness) estiff = ept->stiffness[(size_t)rc.jid*P.env_pad + env];
          if (ept->damping) edamp = ept->damping[(size_t)rc.da*P.env_pad + env];
          if (ept->lin) {
            const float *l = ept->lin + (size_t)6*rc.jid*P.env_pad + env;
            eKq = l[0]; eKqd = l[P.env_pad]; eKqU = l[3*P.env_pad]; eKqdU = l[4*P.env_pad];
          }
          if (ept->gain && rc.wave_act >= 0) ewgain = ept->gain[(size_t)rc.wave_act*P.env_pad + env];
        }
        FB_PIN_F(estiff); FB_PIN_F(edamp);
        FB_PIN_F(eKq); FB_PIN_F(eKqd); FB_PIN_F(eKqU); FB_PIN_F(eKqdU); FB_PIN_F(ewgain);
      }
      if (SPLIT) { pb = block(b); pg = gblock(b); }
      else { pb -= NF*BLK; pg -= GNF*BLK; }
      const int jtype = rc.jtype, flags = rc.flags;
      float cx[10], cxv[6];
FB_UNROLL
      for (int k = 0; k < 10; k++) cx[k] = nx[k];
FB_UNROLL
      for (int k = 0; k < 6; k++) cxv[k] = nxv[k];
      if (bn) {
        const float *pn = SPLIT ? gblock(bn) : pg - GNF*BLK;
FB_UNROLL
        for (int k = 0; k < 6; k++) nx[k] = fb_ld_scr(pn + (FG_W + k)*BLK);
        nx[6] = fb_ld_scr(pn + FG_Q*BLK); nx[7] = fb_ld_scr(pn + FG_QD*BLK);
        nx[8] = fb_ld_scr(pn + FGTC*BLK); nx[9] = fb_ld_scr(pn + FGTU*BLK);
        if (SLIM) {
FB_UNROLL
          for (int k = 0; k < 6; k++) nxv[k] = fb_ld_scr(pn + (FG_V + k)*BLK);
        }
      }
      const Quat q = {pb[(FB_QUAT)*BLK], pb[(FB_QUAT + 1)*BLK], pb[(FB_QUAT + 2)*BLK], pb[(FB_QUAT + 3)*BLK]};
      float R[9], v[6], fx[6];
      q_mat(q, R);
FB_UNROLL
      for (int k = 0; k < 6; k++) { v[k] = SLIM ? cxv[k] : pb[(FB_VEL + k)*BLK]; fx[k] = cx[k]; }
      /* rigid-body inertia about the anchor */
      const float mass = rc.mass;
      float h[3], Iw[6];
      m_rot(R, rc.hloc[0], rc.hloc[1], rc.hloc[2], h);
      if (MODE == 2) {
        /* contact forces of this body's candidates: world force at the contact point */
        for (int fc = rc.bc0; fc < rc.bc1; fc++) {
          if (!fb_bit128(hany, fc)) continue;
          const float *pc_ = ncand(fc);
          const int on = fb_bit128(hm, fc);
          float Fw[3], rr[3], cr[3];
FB_UNROLL
          for (int k = 0; k < 3; k++) {
            Fw[k] = on ? fb_ld_scr(pc_ + (NC_RES + k)*BLK) : 0.f;
            rr[k] = on ? fb_ld_scr(pc_ + (NC_R + k)*BLK) - h[k] : 0.f;
          }
          v_cross(rr, Fw, cr);
FB_UNROLL
          for (int k = 0; k < 3; k++) { fx[k] += Fw[k]; fx[3 + k] += cr[k]; }
        }
      }
      if (LEAN || (flags & FT_AXISYM)) {
        /* Iw = Ia 1 + dI n n', n = R n_body */
        float n[3];
        m_rot(R, rc.Ib[2], rc.Ib[3], rc.Ib[4], n);
        const float ia = rc.Ib[0], d0 = rc.Ib[1]*n[0], d1 = rc.Ib[1]*n[1], d2 = rc.Ib[1]*n[2];
        Iw[0] = ia + d0*n[0]; Iw[1] = ia + d1*n[1]; Iw[2] = ia + d2*n[2];
        Iw[3] = d0*n[1]; Iw[4] = d0*n[2]; Iw[5] = d1*n[2];
      } else {
        /* Iw = R Ib R' */
        float T[9];
FB_UNROLL
        for (int i = 0; i < 3; i++) {
          float ri[3] = {R[3*i], R[3*i+1], R[3*i+2]}, t[3];
          sym_mul(rc.Ib, ri, t);
          T[3*i] = t[0]; T[3*i+1] = t[1]; T[3*i+2] = t[2];       /* row i of R Ib */
        }
        Iw[0] = T[0]*R[0] + T[1]*R[1] + T[2]*R[2];
        Iw[1] = T[3]*R[3] + T[4]*R[4] + T[5]*R[5];
        Iw[2] = T[6]*R[6] + T[7]*R[7] + T[8]*R[8];
        Iw[3] = T[0]*R[3] + T[1]*R[4] + T[2]*R[5];
        Iw[4] = T[0]*R[6] + T[1]*R[7] + T[2]*R[8];
        Iw[5] = T[3]*R[6] + T[4]*R[7] + T[5]*R[8];
      }
      ArtInertia I;
      const float hh = h[0]*h[0] + h[1]*h[1] + h[2]*h[2];
      I.A[0] = Iw[0] + mass*(hh - h[0]*h[0]); I.A[1] = Iw[1] + mass*(hh - h[1]*h[1]);
      I.A[2] = Iw[2] + mass*(hh - h[2]*h[2]);
      I.A[3] = Iw[3] - mass*h[0]*h[1]; I.A[4] = Iw[4] - mass*h[0]*h[2]; I.A[5] = Iw[5] - mass*h[1]*h[2];
      I.H[0] = 0.f; I.H[1] = -mass*h[2]; I.H[2] = mass*h[1];
      I.H[3] = mass*h[2]; I.H[4] = 0.f; I.H[5] = -mass*h[0];
      I.H[6] = -mass*h[1]; I.H[7] = mass*h[0]; I.H[8] = 0.f;
      I.M[0] = mass; I.M[1] = mass; I.M[2] = mass; I.M[3] = 0.f; I.M[4] = 0.f; I.M[5] = 0.f;
      /* bias force  v x* (I v) - applied wrench (force F, torque T at the com) */
      float pA[6];
      {
        float wxh[3], mom[3], L[3], t[3], c1[3], c2[3];
        v_cross(v, h, wxh);
FB_UNROLL
        for (int k = 0; k < 3; k++) mom[k] = mass*(v[3 + k] + wxh[k]);
        sym_mul(Iw, v, L);
        v_cross(h, mom, t);
FB_UNROLL
        for (int k = 0; k < 3; k++) L[k] += t[k];
        v_cross(v, L, c1);
        v_cross(v + 3, mom, c2);
        v_cross(h, fx, t);                        /* h x F */
FB_UNROLL
        for (int k = 0; k < 3; k++) pA[k] = c1[k] + c2[k] - (fx[3 + k] + t[k]);
        v_cross(v, mom, c1);
FB_UNROLL
        for (int k = 0; k < 3; k++) pA[3 + k] = c1[k] - fx[k];
      }
      if (flags & FT_ADD_CARRY) {
FB_UNROLL
        for (int k = 0; k < 6; k++) { I.A[k] += C.A[k]; I.M[k] += C.M[k]; pA[k] += pc[k]; }
FB_UNROLL
        for (int k = 0; k < 9; k++) I.H[k] += C.H[k];
      }
      if (flags & FT_HAS_SLOT) {
        const float *so = slot(rc.slot);
FB_UNROLL
        for (int k = 0; k < 6; k++) { I.A[k] += sl_ld(so, k); I.M[k] += sl_ld(so, 15 + k); pA[k] += sl_ld(so, 21 + k); }
FB_UNROLL
        for (int k = 0; k < 9; k++) I.H[k] += sl_ld(so, 6 + k);
      }
      if (jtype == FB_JNT_FREE) {
        /* floating root: I a + pA = 0 for the (gravity-free frame) acceleration */
        float K[6][6], rhs[6];
        K[0][0] = I.A[0]; K[1][1] = I.A[1]; K[2][2] = I.A[2];
        K[1][0] = I.A[3]; K[2][0] = I.A[4]; K[2][1] = I.A[5];
        K[3][3] = I.M[0]; K[4][4] = I.M[1]; K[5][5] = I.M[2];
        K[4][3] = I.M[3]; K[5][3] = I.M[4]; K[5][4] = I.M[5];
FB_UNROLL
        for (int i = 0; i < 3; i++)
FB_UNROLL
          for (int j = 0; j < 3; j++) K[3 + j][i] = I.H[3*i + j];
FB_UNROLL
        for (int k = 0; k < 6; k++) rhs[k] = -pA[k];
        solve6(K, rhs, aroot);
        continue;
      }
      if (jtype >= 0) {
        const float qj = cx[6], qd = cx[7];
        float ax[3], U[6], c[6], tau, trq;
        m_rot(R, rc.axis[0], rc.axis[1], rc.axis[2], ax);
        if (LEAN || (flags & FT_ACT_SIMPLE)) {
          float tc = cx[8], tu = cx[9];
          if (!LEAN && seqk) seq_constants(rc, seqk, &tc, &tu);
          tau = tc + (ENVP ? eKq : rc.Kq)*qj + (ENVP ? eKqd : rc.Kqd)*qd;
          if (flags & FT_HAS_WAVE) {
            float ph = 6.283185307179586f*rc.wfreq*time - rc.wlag + env_phase;
            float cw = rc.woff + rc.wamp*sinf(ph);
            tau += (ENVP ? ewgain : rc.wgain)*cw;
            if (store_ctrl) P.ctrl[(size_t)env*m.nu + rc.wave_act] = cw;
          }
          trq = tau - (tu + (ENVP ? eKqU : rc.KqU)*qj + (ENVP ? eKqdU : rc.KqdU)*qd);
        } else {
          actuation_generic(rc, qj, qd, time, store_ctrl, seqk, &tau, &trq);
        }
        if ((ENVP ? estiff : rc.stiffness) != 0.f) {
          /* spring reference of this step: a row of the control sequence (on-device CPG), else held */
          const float ref = (!LEAN && seqk && FT_SREF(flags) >= 0) ? seqk[(long long)(m.nu + FT_SREF(flags))*P.env_pad]
                                                           : P.qpos_spring[(size_t)env*m.nq + rc.qa];
          tau -= (ENVP ? estiff : rc.stiffness)*(qj - ref);
        }
        tau -= (ENVP ? edamp : rc.damping)*qd;
        if (MODE == 2) tau += fb_ld_scr(nblock(b) + NB_TAUC*BLK);
        float d, u;
        float aq[3] = {ax[0]*qd, ax[1]*qd, ax[2]*qd};
        if (LEAN || jtype == FB_JNT_HINGE) {
          sym_mul(I.A, ax, U);
          ht_mul(I.H, ax, U + 3);
          d = ax[0]*U[0] + ax[1]*U[1] + ax[2]*U[2];
          u = tau - (ax[0]*pA[0] + ax[1]*pA[1] + ax[2]*pA[2]);
          v_cross(v, aq, c);
          v_cross(v + 3, aq, c + 3);
        } else {
          h_mul(I.H, ax, U);
          sym_mul(I.M, ax, U + 3);
          d = ax[0]*U[3] + ax[1]*U[4] + ax[2]*U[5];
          u = tau - (ax[0]*pA[3] + ax[1]*pA[4] + ax[2]*pA[5]);
          c[0] = c[1] = c[2] = 0.f;
          v_cross(v, aq, c + 3);
        }
        d += MODE == 1 ? rc.armature : rc.armature + hdt*(ENVP ? edamp : rc.damping);
        const float dinv = fb_rcp(d);
        /* Ia = I - U U'/d */
        sym_rank1(I.A, U, dinv);
        sym_rank1(I.M, U + 3, dinv);
FB_UNROLL
        for (int i = 0; i < 3; i++) {
          const float ui = dinv*U[i];
FB_UNROLL
          for (int j = 0; j < 3; j++) I.H[3*i + j] -= ui*U[3 + j];
        }
        /* pa = pA + Ia c + U u/d */
        float t0[3], t1[3];
        const float ud = u*dinv;
        sym_mul(I.A, c, t0); h_mul(I.H, c + 3, t1);
FB_UNROLL
        for (int k = 0; k < 3; k++) pA[k] += t0[k] + t1[k] + U[k]*ud;
        ht_mul(I.H, c, t0); sym_mul(I.M, c + 3, t1);
FB_UNROLL
        for (int k = 0; k < 3; k++) pA[3 + k] += t0[k] + t1[k] + U[3 + k]*ud;
        if (MODE == 1) {
          float *pn_ = nblock(b);
FB_UNROLL
          for (int k = 0; k < 6; k++) fb_st_scr(pn_ + (NB_U + k)*BLK, U[k]);
          fb_st_scr(pn_ + NB_UU*BLK, u); fb_st_scr(pn_ + NB_DINV*BLK, dinv);
        } else {
FB_UNROLL
          for (int k = 0; k < 6; k++) fb_st_scr(pg + (FG_W + k)*BLK, U[k]);
          fb_st_scr(pg + FG_U*BLK, u); fb_st_scr(pg + FG_DINV*BLK, dinv); fb_st_scr(pg + FG_TRQ*BLK, trq);
        }
      }
      if (rc.parent == 0) continue;        /* fixed base: nothing above */
      /* move to the parent's anchor and hand over */
      {
        const float *pp = pblock(rc);
        float r[3];
FB_UNROLL
        for (int k = 0; k < 3; k++) r[k] = pb[(FB_ORG + k)*BLK] - pp[(FB_ORG + k)*BLK];
        art_shift(I, pA, r);
      }
      if (flags & FT_TO_CARRY) {
        C = I;
FB_UNROLL
        for (int k = 0; k < 6; k++) pc[k] = pA[k];
      } else {
        float *so = slot(rc.pslot);
        if (flags & FT_FIRST_WRITER) {
FB_UNROLL
          for (int k = 0; k < 6; k++) { sl_st(so, k, I.A[k]); sl_st(so, 15 + k, I.M[k]); sl_st(so, 21 + k, pA[k]); }
FB_UNROLL
          for (int k = 0; k < 9; k++) sl_st(so, 6 + k, I.H[k]);
        } else {
FB_UNROLL
          for (int k = 0; k < 6; k++) { sl_add(so, k, I.A[k]); sl_add(so, 15 + k, I.M[k]); sl_add(so, 21 + k, pA[k]); }
FB_UNROLL
          for (int k = 0; k < 9; k++) sl_add(so, 6 + k, I.H[k]);
        }
      }
    }
  }

  /* ---- pass 3: root -> leaves, accelerations, Euler, joints / xfrc rows, drag */
  FB_MEM int pass_accel(const float *aroot, float *row_joints, float *row_xfrc) {
    return pass_accel_m<0>(aroot, row_joints, row_xfrc);
  }
  /* CON = 1: the joints rows carry the limit forces of the constrained step */
  template <int CON>
  FB_MEM int pass_accel_m(const float *aroot, float *row_joints, float *row_xfrc) {
    const int nb = m.nbody;
    const float hdt = m.timestep;
    float ac[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   /* carry: acceleration of body b-1 */
    int bad = 0;
    float nx[11] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   /* U[6], u, 1/d, trq, q, qd of the next body to visit */
    float nxv[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};     /* SLIM: its velocity */
    const int n_it = SPLIT ? ord_n : nb - 1;
    {
      const float *pn = gblock(SPLIT ? (ord_n > 0 ? ord[0] : 1) : 1);
FB_UNROLL
      for (int k = 0; k < 9; k++) nx[k] = fb_ld_scr(pn + (FG_W + k)*BLK);     /* W, U, DINV, TRQ are contiguous */
      nx[9] = fb_ld_scr(pn + FG_Q*BLK); nx[10] = fb_ld_scr(pn + FG_QD*BLK);
      if (SLIM) {
FB_UNROLL
        for (int k = 0; k < 6; k++) nxv[k] = fb_ld_scr(pn + (FG_V + k)*BLK);
      }
    }
    float *pb = block(1) - NF*BLK;
    float *pg = gblock(1) - GNF*BLK;
    float nap[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};     /* SLIM: acceleration of the parent of the next body when that is a branch child */
    for (int i = 0; i <= n_it; i++) {
      if (SPLIT && i == ord_bnd) split_barrier();      /* the trunk's accelerations are known */
      if (i == n_it) break;
      if (SPLIT && idle) continue;
      const int b = SPLIT ? ord[i] : i + 1;
      const int bn = SPLIT ? (i + 1 < n_it ? ord[i + 1] : 0) : (i + 2 < nb ? i + 2 : 0);
      const FastRec &rc = rec[b];
      FB_PIN_I(rc.jtype); FB_PIN_I(rc.flags); FB_PIN_I(SLIM ? rc.pblk7 : rc.pblk); FB_PIN_I(rc.parent); FB_PIN_I(rc.fj);
      FB_PIN_I(rc.xr); FB_PIN_I(rc.swim);
      FB_PIN_F(rc.lift); FB_PIN_F(rc.height);
FB_UNROLL
      for (int k = 0; k < 3; k++) { FB_PIN_F(rc.hloc[k]); FB_PIN_F(rc.axis[k]); }
FB_UNROLL
      for (int k = 0; k < 6; k++) FB_PIN_F(rc.coef[k]);
      float ecoef[6], ewv[3];                /* ENVP: this environment's drag values, loads issued here */
      if constexpr (ENVP) if (rc.swim >= 0) {
        const FbEnvTables *ept = this->ept;
FB_UNROLL
        for (int k = 0; k < 6; k++) ecoef[k] = ept->coef ? ept->coef[(size_t)(6*rc.swim + k)*P.env_pad + env] : rc.coef[k];
FB_UNROLL
        for (int k = 0; k < 3; k++) ewv[k] = ept->wvel ? ept->wvel[(size_t)k*P.env_pad + env] : m.water_velocity[k];
FB_UNROLL
        for (int k = 0; k < 6; k++) FB_PIN_F(ecoef[k]);
FB_UNROLL
        for (int k = 0; k < 3; k++) FB_PIN_F(ewv[k]);
      }
      if (SPLIT) { pb = block(b); pg = gblock(b); }
      else { pb += NF*BLK; pg += GNF*BLK; }
      const int jtype = rc.jtype, flags = rc.flags;
      float cx[11], cxv[6];
FB_UNROLL
      for (int k = 0; k < 11; k++) cx[k] = nx[k];
FB_UNROLL
      for (int k = 0; k < 6; k++) cxv[k] = nxv[k];
      if (bn) {
        const float *pn = SPLIT ? gblock(bn) : pg + GNF*BLK;
FB_UNROLL
        for (int k = 0; k < 9; k++) nx[k] = fb_ld_scr(pn + (FG_W + k)*BLK);
        nx[9] = fb_ld_scr(pn + FG_Q*BLK); nx[10] = fb_ld_scr(pn + FG_QD*BLK);
        if (SLIM) {
FB_UNROLL
          for (int k = 0; k < 6; k++) nxv[k] = fb_ld_scr(pn + (FG_V + k)*BLK);
        }
      }
      /* a body without an xfrc row keeps the user's wrench: fetched now, stored at the end of the
       * iteration (the slot held U during this step) */
      float uwr[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (rc.xr < 0) {
        const float *gx = P.xfrc_applied + ((size_t)env*m.nbody + b)*6;
FB_UNROLL
        for (int k = 0; k < 6; k++) uwr[k] = gx[k];
      }
      const Quat q = {pb[(FB_QUAT)*BLK], pb[(FB_QUAT + 1)*BLK], pb[(FB_QUAT + 2)*BLK], pb[(FB_QUAT + 3)*BLK]};
      float R[9], v[6], a[6];
      q_mat(q, R);
FB_UNROLL
      for (int k = 0; k < 6; k++) v[k] = SLIM ? cxv[k] : pb[(FB_VEL + k)*BLK];
      if (jtype == FB_JNT_FREE) {
FB_UNROLL
        for (int k = 0; k < 6; k++) a[k] = aroot[k];
        float cr[3], wl[3], w[3];
        v_cross(v, v + 3, cr);
        m_rot_t(R, a[0], a[1], a[2], wl);
FB_UNROLL
        for (int k = 0; k < 3; k++) {
          float vn = rt[7 + k] + hdt*(a[3 + k] + m.grav[k] + cr[k]);
          rt[7 + k] = vn;
          float pn = rt[k] + hdt*vn;
          rt[k] = pn;
          w[k] = rt[10 + k] + hdt*wl[k];
          rt[10 + k] = w[k];
          bad |= !(fabsf(pn) < 1e30f);
        }
        float angle = hdt*v_normalize3(w), sn, cs;
        fb_sincos_half(0.5f*angle, &sn, &cs);
        Quat qr = {cs, w[0]*sn, w[1]*sn, w[2]*sn};
        Quat qn = q_normalize(q_mul(q, qr));
        rt[3] = qn.w; rt[4] = qn.x; rt[5] = qn.y; rt[6] = qn.z;
        bad |= !(fabsf(qn.w) < 1e30f) | !(fabsf(qn.x) < 1e30f) | !(fabsf(qn.y) < 1e30f) | !(fabsf(qn.z) < 1e30f);
      } else {
        float ap[6] = {0.f, 0.f, 0.f, -m.grav[0], -m.grav[1], -m.grav[2]};
        float r[3] = {0.f, 0.f, 0.f}, cr[3];
        if (rc.parent > 0) {
          const float *pp = pblock(rc);
FB_UNROLL
          for (int k = 0; k < 3; k++) r[k] = pb[(FB_ORG + k)*BLK] - pp[(FB_ORG + k)*BLK];
          if (flags & FT_TO_CARRY) {
FB_UNROLL
            for (int k = 0; k < 6; k++) ap[k] = ac[k];
          } else if (SLIM) {
FB_UNROLL
            for (int k = 0; k < 6; k++) ap[k] = nap[k];
          } else {
            const float *so = slot(rc.pslot);
FB_UNROLL
            for (int k = 0; k < 6; k++) ap[k] = sl_ld(so, k);
          }
        }
        v_cross(ap, r, cr);
FB_UNROLL
        for (int k = 0; k < 3; k++) { a[k] = ap[k]; a[3 + k] = ap[3 + k] + cr[k]; }
        if (jtype >= 0) {
          const float qj = cx[9], qd = cx[10];
          float ax[3], U[6];
          m_rot(R, rc.axis[0], rc.axis[1], rc.axis[2], ax);
FB_UNROLL
          for (int k = 0; k < 6; k++) U[k] = cx[k];
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
          float ua = U[0]*a[0] + U[1]*a[1] + U[2]*a[2] + U[3]*a[3] + U[4]*a[4] + U[5]*a[5];
          const float qdd = (cx[6] - ua)*cx[7];
          if (LEAN || jtype == FB_JNT_HINGE) { a[0] += ax[0]*qdd; a[1] += ax[1]*qdd; a[2] += ax[2]*qdd; }
          else { a[3] += ax[0]*qdd; a[4] += ax[1]*qdd; a[5] += ax[2]*qdd; }
          const float qdn = qd + hdt*qdd, qn = qj + hdt*qdn;
          fb_st_scr(pg + FG_QD*BLK, qdn);
          fb_st_scr(pg + FG_Q*BLK, qn);
          bad |= !(fabsf(qn) < 1e30f);
          /* joints row: physics.py:481-524 (new position/velocity, forces of the old state) */
          if (rc.fj >= 0) {
            const long long ev = P.env_pad*FB_VEC_JOINTS;
            const int cp = m.col_jpos, cv = m.col_jvel, ct = m.col_jtrq, cols = m.joint_cols;
            float *row = row_joints + (long long)((cols/2)*rc.fj)*ev;   /* 8-byte vectors, coalesced across the warp */
            const float trq = cx[8]*m.inv_torques, jv = qdn*m.inv_angvel;
            const float lf = CON ? fb_ld_scr(nblock(b) + NB_LIMF*BLK)*m.inv_torques : 0.f;
            const int cl = CON ? m.col_jlim : -1;
            /* The other columns of the row (physics.py:481-524 leaves 14 of the 18 untouched) are
             * zero in the log from its allocation on and no kernel writes them; the limit-force pair
             * is written by constrained steps, and here only over a row that may hold one. */
            if (LEAN || m.X.jrow_std) {
              /* farms layout: 18 columns, position 0, velocity 1, torque 11, limit force 16 */
              fb_st2(row, qn, jv);
              fb_st2(row + 5*ev, 0.f, trq);
              if (CON || zfill) fb_st2(row + 8*ev, lf, 0.f);
            } else {
              const int cz = CON || zfill ? m.col_jlim : -1;
#define FB_JCOL(c_) ((c_) == cp ? qn : ((c_) == cv ? jv : ((c_) == ct ? trq : ((c_) == cl ? lf : 0.f))))
#define FB_JHAS(c_) ((c_) == cp || (c_) == cv || (c_) == ct || (c_) == cz)
              for (int c = 0; c < cols; c += 2)
                if (FB_JHAS(c) || FB_JHAS(c + 1)) fb_st2(row + (c/2)*ev, FB_JCOL(c), FB_JCOL(c + 1));
#undef FB_JHAS
#undef FB_JCOL
            }
          }
        }
      }
FB_UNROLL
      for (int k = 0; k < 6; k++) ac[k] = a[k];
      if (flags & FT_HAS_SLOT) {
        float *so = slot(rc.slot);
FB_UNROLL
        for (int k = 0; k < 6; k++) sl_st(so, k, a[k]);
      }
      if (SLIM && b + 1 < nb) {
        const FastRec &rn = rec[b + 1];
        if (!(rn.flags & FT_TO_CARRY) && rn.parent > 0) {
          if (rn.parent == b) {             /* (cannot happen: a child of b that follows it is a carry child) */
FB_UNROLL
            for (int k = 0; k < 6; k++) nap[k] = a[k];
          } else {
            const float *so = slot(rn.pslot);
FB_UNROLL
            for (int k = 0; k < 6; k++) nap[k] = sl_ld(so, k);
          }
        }
      }
      /* xfrc row + the wrench applied during the next step (drag.pyx:152-268, 3.4) */
      if (rc.xr >= 0) {
        float F[3] = {0.f, 0.f, 0.f}, Tq[3] = {0.f, 0.f, 0.f}, wf[3] = {0.f, 0.f, 0.f}, wt[3] = {0.f, 0.f, 0.f};
        if (m.water_drag && rc.swim >= 0) {
          float h[3], cr[3], lin[3], vl[3], wl[3], uw[3], buoy[3] = {0.f, 0.f, 0.f};
          m_rot(R, rc.hloc[0], rc.hloc[1], rc.hloc[2], h);
          const float pz = (rootpos[2] + pb[(FB_ORG + 2)*BLK] + h[2])*m.inv_meters;
          if (!(pz > m.water_surface)) {                 /* drag.pyx:192-194 */
            v_cross(v, h, cr);
FB_UNROLL
            for (int k = 0; k < 3; k++) lin[k] = v[3 + k] + cr[k];
            m_rot_t(R, lin[0]*m.inv_velocity, lin[1]*m.inv_velocity, lin[2]*m.inv_velocity, vl);
            m_rot_t(R, v[0]*m.inv_angvel, v[1]*m.inv_angvel, v[2]*m.inv_angvel, wl);
            if (m.water_buoyancy && rc.lift > 0.f && pz < m.water_surface) {
              float frac = fminf(fmaxf(m.water_surface - pz, 0.f)/rc.height, 1.f);
              m_rot_t(R, 0.f, 0.f, rc.lift*frac, buoy);
            }
            if (ENVP) m_rot_t(R, ewv[0], ewv[1], ewv[2], uw);
            else m_rot_t(R, m.water_velocity[0], m.water_velocity[1], m.water_velocity[2], uw);
FB_UNROLL
            for (int k = 0; k < 3; k++) {
              float vv = vl[k] - uw[k], w = wl[k];
              float sv = vv < 0.f ? -vv*vv : vv*vv, sw = w < 0.f ? -w*w : w*w;
              F[k] = sv*m.water_viscosity*(ENVP ? ecoef[k] : rc.coef[k]) + buoy[k];
              Tq[k] = sw*(ENVP ? ecoef[3 + k] : rc.coef[3 + k]);
            }
            m_rot(R, F[0], F[1], F[2], wf);
            m_rot(R, Tq[0], Tq[1], Tq[2], wt);
FB_UNROLL
            for (int k = 0; k < 3; k++) { wf[k] *= m.newtons; wt[k] *= m.torques; }
          }
        }
        const long long ev = P.env_pad*FB_VEC_XFRC;
        float *row = row_xfrc + (long long)(3*rc.xr)*ev;
        fb_st2(row, F[0], F[1]); fb_st2(row + ev, F[2], Tq[0]); fb_st2(row + 2*ev, Tq[1], Tq[2]);
FB_UNROLL
        for (int k = 0; k < 3; k++) { fb_st_scr(pg + (FG_W + k)*BLK, wf[k]); fb_st_scr(pg + (FG_W + 3 + k)*BLK, wt[k]); }
      } else {
        /* user-applied wrench: persistent, re-read (the slot held U during this step) */
FB_UNROLL
        for (int k = 0; k < 6; k++) fb_st_scr(pg + (FG_W + k)*BLK, uwr[k]);
      }
    }
    return bad;
  }

  /* Returns the number of steps taken here (n_steps unless a constraint appeared). */
  FB_MEM int run(int coop, int lane) { return run_t<0>(coop, lane, 1); }
  /* SYNC = 1: the warps of a block meet at a barrier before every pass.  They run the same
   * instruction stream, so they then walk the same loop bodies at the same time and share their
   * instruction-cache lines (the three body loops are ~30 KB each, the L1.5 I-cache 32 KB: warps at
   * unrelated program positions miss in it all the time -- 20 % of the stall samples with eight
   * resident warps).  Every thread of the block takes every iteration: an environment that hands
   * over (or a thread beyond the batch, valid = 0) idles through the rest instead of leaving. */
  template <int SYNC>
  FB_MEM int run_t(int coop, int lane, int valid) {
    if (valid) load_state(coop, lane);
    const size_t e = (size_t)env;
    const int n = P.n_steps;
    int kdone = n, dead = !valid;
    long long row = P.it0 % P.ring;       /* one 64-bit division per launch, not per step */
    for (int k = 0; k < n; k++) {
      row = row + 1 == P.ring ? 0 : row + 1;
      float *row_links = fb_log_row(P.log_links, row, m.n_links*20, P.env_pad, FB_VEC_LINKS, e);
      float *row_joints = fb_log_row(P.log_joints, row, m.n_joints*m.joint_cols, P.env_pad, FB_VEC_JOINTS, e);
      float *row_contacts = fb_log_row(P.log_contacts, row, m.n_contacts*12, P.env_pad, FB_VEC_CONTACTS, e);
      float *row_xfrc = fb_log_row(P.log_xfrc, row, m.n_xfrc*6, P.env_pad, FB_VEC_XFRC, e);
      const float time = (float)this->episode_it(P.it0 + k)*m.timestep;
      zfill = log_row_dirty(P.it0 + k + 1);
      fb_block_sync<SYNC>();
      if (!dead && pass_poses(row_links)) { kdone = k; dead = 1; }
      if (!SYNC && dead) break;
      if (!dead && rec[1].jtype == FB_JNT_FREE) { rt[3] = rqn[0]; rt[4] = rqn[1]; rt[5] = rqn[2]; rt[6] = rqn[3]; }
      float aroot[6] = {0.f, 0.f, 0.f, -m.grav[0], -m.grav[1], -m.grav[2]};
      const float *seqk = P.ctrl_seq ? P.ctrl_seq + ((size_t)(P.seq_pos + k)*P.seq_stride)*P.env_pad + e : 0;
      fb_block_sync<SYNC>();
      if (!dead) pass_inertia(time, aroot, k == n - 1 && m.n_wc > 0, seqk);   /* ctrl is left as the team path leaves it */
      fb_block_sync<SYNC>();
      if (dead) continue;
      int bad = pass_accel(aroot, row_joints, row_xfrc);
      /* the contacts rows are what the log holds already unless a constrained step wrote this ring
       * row before */
      if (zfill) zero_contacts(row_contacts);
      if (bad) FB_FLAG_OR(P.flags + env, FB_FLAG_NONFINITE);
    }
    if (!valid) return n;
    if (P.ctrl_seq && kdone == n) store_seq_end(n);
    store_state(P.it0 + kdone, coop, lane);
    return kdone;
  }

  /* SPLIT: run_t's protocol for a block whose warps step the SAME 32 environments, each its own
   * bodies (split_setup).  Every thread takes every barrier; warp 0 owns the root state, the state
   * I/O and the hand-over bookkeeping; a lane leaves the step when ANY warp saw one of its bodies at
   * a limit or inside a plane bound. */
  FB_MEM int run_split(int coop, int lane, int valid) {
    if (role == 0 && valid) load_state(coop, lane);
    FB_BLOCK_BARRIER();
    const size_t e = (size_t)env;
    const int n = P.n_steps;
    int kdone = n, dead = !valid;
    long long row = P.it0 % P.ring;
    for (int k = 0; k < n; k++) {
      row = row + 1 == P.ring ? 0 : row + 1;
      float *row_links = fb_log_row(P.log_links, row, m.n_links*20, P.env_pad, FB_VEC_LINKS, e);
      float *row_joints = fb_log_row(P.log_joints, row, m.n_joints*m.joint_cols, P.env_pad, FB_VEC_JOINTS, e);
      float *row_contacts = fb_log_row(P.log_contacts, row, m.n_contacts*12, P.env_pad, FB_VEC_CONTACTS, e);
      float *row_xfrc = fb_log_row(P.log_xfrc, row, m.n_xfrc*6, P.env_pad, FB_VEC_XFRC, e);
      const float time = (float)this->episode_it(P.it0 + k)*m.timestep;
      zfill = log_row_dirty(P.it0 + k + 1);
      if (role == 0) sflag[0] = 0;
      FB_BLOCK_BARRIER();
      idle = dead;
      const int act = pass_poses(row_links);
      if (!dead && act) sflag[0] = 1;
      FB_BLOCK_BARRIER();
      if (!dead && sflag[0]) { kdone = k; dead = 1; }
      idle = dead;
      if (role == 0 && !dead && rec[1].jtype == FB_JNT_FREE) { rt[3] = rqn[0]; rt[4] = rqn[1]; rt[5] = rqn[2]; rt[6] = rqn[3]; }
      float aroot[6] = {0.f, 0.f, 0.f, -m.grav[0], -m.grav[1], -m.grav[2]};
      const float *seqk = P.ctrl_seq ? P.ctrl_seq + ((size_t)(P.seq_pos + k)*P.seq_stride)*P.env_pad + e : 0;
      pass_inertia(time, aroot, k == n - 1 && m.n_wc > 0, seqk);
      FB_BLOCK_BARRIER();
      const int bad = pass_accel(aroot, row_joints, row_xfrc);
      if (!dead) {
        if (zfill && role == 0) zero_contacts(row_contacts);
        if (bad) FB_FLAG_OR(P.flags + env, FB_FLAG_NONFINITE);
      }
    }
    FB_BLOCK_BARRIER();
    if (role != 0 || !valid) return n;
    if (P.ctrl_seq && kdone == n) store_seq_end(n);
    store_state(P.it0 + kdone, coop, lane);
    return kdone;
  }
};

#endif /* FB_FAST_H_ */
