/*
 * fb_device.h -- the fused FARMS step: MuJoCo-subset forward dynamics, soft
 * constraints, semi-implicit Euler, farms sensor log rows and the swimming
 * drag model, for ONE environment cooperatively executed by a TEAM of lanes
 * (TEAM = 8, 16 or 32 lanes of one warp; the environment's working set lives
 * in shared memory as component-major SoA arrays, see DevLayout).
 *
 * Algorithm references (SURVEY.md Appendix A restates the third-party MuJoCo
 * pipeline; the farms parts follow the reference source directly):
 *   step order            mj_step via farms_mujoco/simulation/simulation.py:156
 *   log rows              farms_mujoco/simulation/physics.py:449-524
 *   contact aggregation   farms_mujoco/sensors/sensors.pyx:20-190
 *   drag / buoyancy       farms_mujoco/swimming/drag.pyx:152-268,389-411
 *   hook order            farms_mujoco/simulation/task.py:168-186
 *
 * The file compiles in two ways:
 *   - nvcc (sm_100a): the product.  Team primitives are warp shuffles,
 *     __ballot_sync and __syncwarp on the team's lane mask.
 *   - g++ with -DFB_HOST_EMU (tests/emu only): TEAM = 1, primitives collapse to
 *     identities.  This is a unit-test harness for the arithmetic and indexing
 *     in fp32 on the CPU-only development box; it is never loaded by the
 *     product path.
 */
#ifndef FB_DEVICE_H_
#define FB_DEVICE_H_

#include "fb_model.h"

#ifdef FB_HOST_EMU
#include <cmath>
#define FB_DEV static inline
#define FB_UNROLL
#define FB_MEM inline
#define FB_LDG(p) (*(p))
static inline float fb_rsqrt(float x) { return 1.0f/sqrtf(x); }
static inline void fb_sincos(float x, float *s, float *c) { *s = sinf(x); *c = cosf(x); }
#else
#define FB_DEV __device__ __forceinline__
#define FB_UNROLL _Pragma("unroll")
#define FB_MEM __device__ __forceinline__
#define FB_LDG(p) __ldg(p)
__device__ __forceinline__ float fb_rsqrt(float x) { return 1.0f/sqrtf(x); }
__device__ __forceinline__ void fb_sincos(float x, float *s, float *c) { sincosf(x, s, c); }
#endif

#ifdef FB_HOST_EMU
#include <pthread.h>
#include <cstring>
#define FB_POPC(x) __builtin_popcount(x)
#define FB_FLAG_OR(ptr, bit) __atomic_fetch_or((ptr), (bit), __ATOMIC_RELAXED)
/* SPLIT variants under the test harness: the warps of a block are host threads (one lane each)
 * that meet at this barrier; NULL outside such a run */
static pthread_barrier_t *fb_emu_bar = 0;
#define FB_BLOCK_BARRIER() do { if (fb_emu_bar) pthread_barrier_wait(fb_emu_bar); } while (0)
static inline float fb_u2f(unsigned u) { float f; std::memcpy(&f, &u, 4); return f; }
static inline unsigned fb_f2u(float f) { unsigned u; std::memcpy(&u, &f, 4); return u; }
#else
#define FB_POPC(x) __popc(x)
#define FB_FLAG_OR(ptr, bit) atomicOr((ptr), (bit))
#define FB_BLOCK_BARRIER() __syncthreads()
__device__ __forceinline__ float fb_u2f(unsigned u) { return __uint_as_float(u); }
__device__ __forceinline__ unsigned fb_f2u(float f) { return __float_as_uint(f); }
#endif

#define MI(name, i) FB_LDG(m.I + m.o.name + (i))
#define MF(name, i) FB_LDG(m.F + m.o.name + (i))

/* flags (FbStateView.flags_dev) */
#define FB_FLAG_NONFINITE 1
#define FB_FLAG_CONTACT_OVERFLOW 2
#define FB_FLAG_SOLVER 4

/* per-environment global pointers */
struct EnvPtrs {
  float *qpos, *qvel, *ctrl, *xfrc_applied, *qpos_spring;
  float env_phase;
  int *flags;
  /* derived (FbDerivedView) */
  float *d_xpos, *d_xquat, *d_xipos, *d_linvel, *d_angvel, *d_actf, *d_limf, *d_qacc;
  int *d_ncon, *d_con_cand;
  float *d_con_dist, *d_con_pos, *d_con_frame, *d_con_force;
  /* solver scratch */
  float *J3;     /* [3*maxcon][nv] contact-frame rows of the point Jacobian */
  float *efc;    /* [5][maxefc]: aref, D, res, jp, force */
  float *prod3;  /* [2][3*maxcon] */
  /* log rows of this step: element (item, col) of a kind with C columns stored in vectors of
   * V lives at row[(item*(C/V) + col/V)*ev + col%V], ev = env_pad*V (FbLogView) */
  float *row_links, *row_joints, *row_contacts, *row_xfrc;
  long long ev_links, ev_joints, ev_contacts, ev_xfrc;
  /* per-environment parameters (fb_set_env_param), already offset by the environment: value c of
   * item i at ep_*[(i*k + c)*ep_pad]; NULL = the model's value */
  const float *ep_stiffness, *ep_damping, *ep_coef, *ep_wvel;
  long long ep_pad;
  /* sliding friction of candidate c at fric[c*fric_stride]: this environment's column of the
   * FB_ENV_CAND_FRICTION table (stride env_pad), else the model's cand_friction (stride 1) */
  const float *fric;
  int fric_stride;
};

/* vector widths of the device log (floats of one row stored contiguously per environment) */
#define FB_VEC_LINKS 4
#define FB_VEC_JOINTS 2
#define FB_VEC_CONTACTS 4
#define FB_VEC_XFRC 2

/* ------------------------------------------------------------ team ops */
template <int TEAM> struct TeamOps {
#ifdef FB_HOST_EMU
  static inline void sync(unsigned) {}
  static inline float sum(unsigned, float v) { return v; }
  static inline float max(unsigned, float v) { return v; }
  static inline float min(unsigned, float v) { return v; }
  static inline unsigned ballot(unsigned, int, int pred) { return pred ? 1u : 0u; }
#else
  static __device__ __forceinline__ void sync(unsigned mask) { __syncwarp(mask); }
  static __device__ __forceinline__ float sum(unsigned mask, float v) {
#pragma unroll
    for (int o = TEAM/2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
    return v;
  }
  static __device__ __forceinline__ float max(unsigned mask, float v) {
#pragma unroll
    for (int o = TEAM/2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(mask, v, o));
    return v;
  }
  static __device__ __forceinline__ float min(unsigned mask, float v) {
#pragma unroll
    for (int o = TEAM/2; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(mask, v, o));
    return v;
  }
  /* team-local ballot: bit i = predicate of team lane i */
  static __device__ __forceinline__ unsigned ballot(unsigned mask, int base, int pred) {
    unsigned b = __ballot_sync(mask, pred);
    return TEAM == 32 ? b : ((b >> base) & ((1u << TEAM) - 1u));
  }
#endif
};

/* --------------------------------------------------------- small algebra */
struct Quat { float w, x, y, z; };

FB_DEV Quat q_mul(Quat a, Quat b) {
  Quat r;
  r.w = a.w*b.w - a.x*b.x - a.y*b.y - a.z*b.z;
  r.x = a.w*b.x + a.x*b.w + a.y*b.z - a.z*b.y;
  r.y = a.w*b.y - a.x*b.z + a.y*b.w + a.z*b.x;
  r.z = a.w*b.z + a.x*b.y - a.y*b.x + a.z*b.w;
  return r;
}
FB_DEV Quat q_normalize(Quat q) {
  float n2 = q.w*q.w + q.x*q.x + q.y*q.y + q.z*q.z;
  if (n2 < 1e-30f) { Quat i = {1.f, 0.f, 0.f, 0.f}; return i; }
  float s = fb_rsqrt(n2);
  Quat r = {q.w*s, q.x*s, q.y*s, q.z*s};
  return r;
}
/* v' = q v q* for a unit quaternion: v + w t + u x t with t = 2 u x v */
FB_DEV void q_rot(Quat q, const float *v, float *o) {
  float tx = 2.f*(q.y*v[2] - q.z*v[1]), ty = 2.f*(q.z*v[0] - q.x*v[2]), tz = 2.f*(q.x*v[1] - q.y*v[0]);
  o[0] = v[0] + q.w*tx + (q.y*tz - q.z*ty);
  o[1] = v[1] + q.w*ty + (q.z*tx - q.x*tz);
  o[2] = v[2] + q.w*tz + (q.x*ty - q.y*tx);
}
FB_DEV void q_mat(Quat q, float *R) {
  float w = q.w, x = q.x, y = q.y, z = q.z;
  R[0] = w*w + x*x - y*y - z*z; R[1] = 2*(x*y - w*z);         R[2] = 2*(x*z + w*y);
  R[3] = 2*(x*y + w*z);         R[4] = w*w - x*x + y*y - z*z; R[5] = 2*(y*z - w*x);
  R[6] = 2*(x*z - w*y);         R[7] = 2*(y*z + w*x);         R[8] = w*w - x*x - y*y + z*z;
}
FB_DEV void m_rot(const float *R, float x, float y, float z, float *o) {
  o[0] = R[0]*x + R[1]*y + R[2]*z;
  o[1] = R[3]*x + R[4]*y + R[5]*z;
  o[2] = R[6]*x + R[7]*y + R[8]*z;
}
FB_DEV void m_rot_t(const float *R, float x, float y, float z, float *o);
FB_DEV void v_cross(const float *a, const float *b, float *o);
FB_DEV float v_normalize3(float *v);
/* mjc_PlaneCylinder: point k (0: the lowest rim point, 1: the rim point at the other end, 2 / 3: the
 * two points that make a triangle with it on the lower rim) of a cylinder (axis, x axis, radius,
 * half length; centre at distance dist0 from the plane along n).  Returns the point's distance from
 * the plane; p = the point relative to the centre. */
FB_DEV float fb_plane_cylinder_point(const float *n, const float *axis_in, const float *xaxis, float radius,
                                     float half, int k, float dist0, float *p) {
  float axis[3] = {axis_in[0], axis_in[1], axis_in[2]}, vec[3], vec1[3];
  float prjaxis = n[0]*axis[0] + n[1]*axis[1] + n[2]*axis[2];
  if (prjaxis > 0.f) { axis[0] = -axis[0]; axis[1] = -axis[1]; axis[2] = -axis[2]; prjaxis = -prjaxis; }
  for (int i = 0; i < 3; i++) vec[i] = axis[i]*prjaxis - n[i];
  const float len = sqrtf(vec[0]*vec[0] + vec[1]*vec[1] + vec[2]*vec[2]);
  if (len >= FB_MINVAL) { for (int i = 0; i < 3; i++) vec[i] *= radius/len; }
  else { for (int i = 0; i < 3; i++) vec[i] = xaxis[i]*radius; }          /* disk parallel to the plane */
  const float prjvec = vec[0]*n[0] + vec[1]*n[1] + vec[2]*n[2];
  for (int i = 0; i < 3; i++) axis[i] *= half;
  prjaxis *= half;
  if (k == 0) { for (int i = 0; i < 3; i++) p[i] = vec[i] + axis[i]; return dist0 + prjaxis + prjvec; }
  if (k == 1) { for (int i = 0; i < 3; i++) p[i] = vec[i] - axis[i]; return dist0 - prjaxis + prjvec; }
  v_cross(vec, axis, vec1);
  v_normalize3(vec1);
  const float sg = k == 2 ? 0.8660254037844386f*radius : -0.8660254037844386f*radius;      /* sqrt(3)/2 */
  for (int i = 0; i < 3; i++) p[i] = sg*vec1[i] + axis[i] - 0.5f*vec[i];
  return dist0 + prjaxis - 0.5f*prjvec;
}

FB_DEV void m_rot_t(const float *R, float x, float y, float z, float *o) {
  o[0] = R[0]*x + R[3]*y + R[6]*z;
  o[1] = R[1]*x + R[4]*y + R[7]*z;
  o[2] = R[2]*x + R[5]*y + R[8]*z;
}
FB_DEV void v_cross(const float *a, const float *b, float *r) {
  float x = a[1]*b[2] - a[2]*b[1], y = a[2]*b[0] - a[0]*b[2], z = a[0]*b[1] - a[1]*b[0];
  r[0] = x; r[1] = y; r[2] = z;
}
/* 10-number spatial inertia times [ang; lin] (mju_mulInertVec) */
FB_DEV void inert_vec(const float *i, const float *v, float *r) {
  r[0] = i[0]*v[0] + i[3]*v[1] + i[4]*v[2] - i[8]*v[4] + i[7]*v[5];
  r[1] = i[3]*v[0] + i[1]*v[1] + i[5]*v[2] + i[8]*v[3] - i[6]*v[5];
  r[2] = i[4]*v[0] + i[5]*v[1] + i[2]*v[2] - i[7]*v[3] + i[6]*v[4];
  r[3] = i[8]*v[1] - i[7]*v[2] + i[9]*v[3];
  r[4] = i[6]*v[2] - i[8]*v[0] + i[9]*v[4];
  r[5] = i[7]*v[0] - i[6]*v[1] + i[9]*v[5];
}
/* vel x_m v (mju_crossMotion) */
FB_DEV void cross_motion(const float *vel, const float *v, float *r) {
  r[0] = -vel[2]*v[1] + vel[1]*v[2];
  r[1] =  vel[2]*v[0] - vel[0]*v[2];
  r[2] = -vel[1]*v[0] + vel[0]*v[1];
  r[3] = -vel[2]*v[4] + vel[1]*v[5] - vel[5]*v[1] + vel[4]*v[2];
  r[4] =  vel[2]*v[3] - vel[0]*v[5] + vel[5]*v[0] - vel[3]*v[2];
  r[5] = -vel[1]*v[3] + vel[0]*v[4] - vel[4]*v[0] + vel[3]*v[1];
}
/* vel x* f (mju_crossForce) */
FB_DEV void cross_force(const float *vel, const float *f, float *r) {
  r[0] = -vel[2]*f[1] + vel[1]*f[2] - vel[5]*f[4] + vel[4]*f[5];
  r[1] =  vel[2]*f[0] - vel[0]*f[2] + vel[5]*f[3] - vel[3]*f[5];
  r[2] = -vel[1]*f[0] + vel[0]*f[1] - vel[4]*f[3] + vel[3]*f[4];
  r[3] = -vel[2]*f[4] + vel[1]*f[5];
  r[4] =  vel[2]*f[3] - vel[0]*f[5];
  r[5] = -vel[1]*f[3] + vel[0]*f[4];
}
FB_DEV float v_normalize3(float *v) {
  float n = sqrtf(v[0]*v[0] + v[1]*v[1] + v[2]*v[2]);
  if (n < 1e-15f) { v[0] = 1.f; v[1] = 0.f; v[2] = 0.f; return n; }
  float s = 1.0f/n;
  v[0] *= s; v[1] *= s; v[2] *= s;
  return n;
}
FB_DEV int pack_idx(int row, int col) { return row*(row + 1)/2 + col; }  /* row >= col */

/* impedance sigmoid (mj getimpedance; SURVEY.md A.7) */
FB_DEV float fb_impedance(const float *solimp, float pos_minus_margin) {
  float dmin = fminf(FB_MAXIMP, fmaxf(FB_MINIMP, solimp[0]));
  float dmax = fminf(FB_MAXIMP, fmaxf(FB_MINIMP, solimp[1]));
  float width = fmaxf(FB_MINVAL, solimp[2]);
  float mid = fminf(FB_MAXIMP, fmaxf(FB_MINIMP, solimp[3]));
  float power = fmaxf(1.0f, solimp[4]);
  if (dmin == dmax || width <= FB_MINVAL) return 0.5f*(dmin + dmax);
  float x = fabsf(pos_minus_margin)/width, y;
  if (x >= 1.f) return dmax;
  if (x <= 0.f) return dmin;
  if (power == 1.f) y = x;
  else if (x <= mid) y = powf(x, power)/powf(mid, power - 1.f);
  else y = 1.f - powf(1.f - x, power)/powf(1.f - mid, power - 1.f);
  return dmin + y*(dmax - dmin);
}
/* K, B, imp, R of one soft-constraint row (mj_makeImpedance) */
FB_DEV void fb_row_params(float timestep, const float *solref_in, const float *solimp,
                          float pos_minus_margin, float diag_approx,
                          float *K, float *B, float *imp, float *R) {
  float sr0 = solref_in[0], sr1 = solref_in[1];
  if (sr0 > 0.f) sr0 = fmaxf(sr0, 2.f*timestep);
  float dmax = fminf(FB_MAXIMP, fmaxf(FB_MINIMP, solimp[1]));
  *imp = fb_impedance(solimp, pos_minus_margin);
  *R = fmaxf(FB_MINVAL, (1.f - *imp)*diag_approx/(*imp));
  if (sr0 > 0.f) {
    *K = 1.f/fmaxf(FB_MINVAL, dmax*dmax*sr0*sr0*sr1*sr1);
    *B = 2.f/fmaxf(FB_MINVAL, dmax*sr0);
  } else {
    *K = -sr0/fmaxf(FB_MINVAL, dmax*dmax);
    *B = -sr1/fmaxf(FB_MINVAL, dmax);
  }
}

/* ===================================================================== */
template <int TEAM> struct FbStep {
  typedef TeamOps<TEAM> T;
  /* bodies per lane held in registers by the subtree-sum phase (nbody <= BPL*TEAM) */
  static const int BPL = TEAM >= 8 ? 2 : 64;
  const DevModel &m;
  float *s;     /* shared floats of this environment */
  int *si;      /* shared ints of this environment */
  EnvPtrs g;
  int lane, base;
  unsigned mask;
  float comx, comy, comz;
  int ncon, nlim;
  int npair_act;   /* active contacts of explicit pairs (two-body rows) */
  int nhard_act;   /* ... of them frictionless: hard normal rows (kind 10) */

  FB_MEM FbStep(const DevModel &m_, float *s_, int *si_, const EnvPtrs &g_, int lane_, int base_,
                unsigned mask_)
      : m(m_), s(s_), si(si_), g(g_), lane(lane_), base(base_), mask(mask_),
        comx(0.f), comy(0.f), comz(0.f), ncon(0), nlim(0), npair_act(0), nhard_act(0) {}

  FB_MEM void sync() { T::sync(mask); }

  /* sliding friction of candidate c: this environment's where FB_ENV_CAND_FRICTION is set (one load
   * without a branch either way: the branch cost the table-free team kernel 1 %) */
  FB_MEM float cand_mu(int c) const { return FB_LDG(g.fric + c*g.fric_stride); }

  /* ------------------------------------------------------------ init */
  FB_MEM void init_world() {
    const int nb = m.nbody;
    if (lane == 0) {
      float *xpos = s + m.L.xpos, *xquat = s + m.L.xquat, *xipos = s + m.L.xipos;
      float *cvel = s + m.L.cvel, *cin = s + m.L.cinert, *xf = s + m.L.xfrc;
      for (int k = 0; k < 3; k++) { xpos[k*nb] = 0.f; xipos[k*nb] = 0.f; }
      xquat[0] = 1.f; xquat[nb] = 0.f; xquat[2*nb] = 0.f; xquat[3*nb] = 0.f;
      for (int k = 0; k < 6; k++) { cvel[k*nb] = 0.f; xf[k*nb] = 0.f; }
      for (int k = 0; k < 10; k++) cin[k*nb] = 0.f;
    }
  }

  /* ------------------------------------------------- A.1 kinematics */
  /* Body frames by pointer jumping instead of a walk over tree depth: every body
   * starts with its transform relative to the parent, then ceil(log2(depth)) rounds
   * compose it with the transform of its 2^r-th ancestor (rigid transforms are
   * associative; the world absorbs).  All lanes work in every round. */
  FB_MEM void kinematics() {
    const int nb = m.nbody, nj = m.njnt, R = m.nround_anc;
    float *qpos = s + m.L.qpos;
    float *mainP = s + m.L.xpos, *mainQ = s + m.L.xquat;
    float *altP = s + m.L.altB, *altQ = s + m.L.altB + 3*nb;
    float *curP = (R & 1) ? altP : mainP, *curQ = (R & 1) ? altQ : mainQ;
    float *nxtP = (R & 1) ? mainP : altP, *nxtQ = (R & 1) ? mainQ : altQ;
    for (int b = lane; b < nb; b += TEAM) {
      float lp[3] = {0.f, 0.f, 0.f};
      Quat lq = {1.f, 0.f, 0.f, 0.f};
      if (b > 0) {
        int jid = MI(body_jnt, b);
        int jtype = jid >= 0 ? MI(jnt_type, jid) : -1;
        if (jtype == FB_JNT_FREE) {
          int qa = MI(jnt_qposadr, jid);
          lp[0] = qpos[qa]; lp[1] = qpos[qa+1]; lp[2] = qpos[qa+2];
          Quat qq = {qpos[qa+3], qpos[qa+4], qpos[qa+5], qpos[qa+6]};
          lq = q_normalize(qq);
          qpos[qa+3] = lq.w; qpos[qa+4] = lq.x; qpos[qa+5] = lq.y; qpos[qa+6] = lq.z;
        } else {
          lp[0] = MF(body_pos, 3*b); lp[1] = MF(body_pos, 3*b+1); lp[2] = MF(body_pos, 3*b+2);
          Quat bq = {MF(body_quat, 4*b), MF(body_quat, 4*b+1), MF(body_quat, 4*b+2),
                     MF(body_quat, 4*b+3)};
          lq = bq;
          if (jid >= 0) {
            float ja[3] = {MF(jnt_axis, 3*jid), MF(jnt_axis, 3*jid+1), MF(jnt_axis, 3*jid+2)};
            float dq = qpos[MI(jnt_qposadr, jid)] - MF(jnt_qpos0, jid);
            if (jtype == FB_JNT_HINGE) {
              float jp[3] = {MF(jnt_pos, 3*jid), MF(jnt_pos, 3*jid+1), MF(jnt_pos, 3*jid+2)};
              float sn, cs, t0[3], t1[3];
              fb_sincos(0.5f*dq, &sn, &cs);
              Quat ql = {cs, ja[0]*sn, ja[1]*sn, ja[2]*sn};
              lq = q_mul(bq, ql);
              q_rot(bq, jp, t0);        /* anchor offset before ... */
              q_rot(lq, jp, t1);        /* ... and after the joint rotation */
              lp[0] += t0[0] - t1[0]; lp[1] += t0[1] - t1[1]; lp[2] += t0[2] - t1[2];
            } else {
              float t0[3];
              q_rot(bq, ja, t0);
              lp[0] += t0[0]*dq; lp[1] += t0[1]*dq; lp[2] += t0[2]*dq;
            }
          }
        }
      }
      curP[b] = lp[0]; curP[nb + b] = lp[1]; curP[2*nb + b] = lp[2];
      curQ[b] = lq.w; curQ[nb + b] = lq.x; curQ[2*nb + b] = lq.y; curQ[3*nb + b] = lq.z;
    }
    sync();
    for (int r = 0; r < R; r++) {
      for (int b = lane; b < nb; b += TEAM) {
        int a = MI(body_anc, r*nb + b);
        Quat qa = {curQ[a], curQ[nb + a], curQ[2*nb + a], curQ[3*nb + a]};
        Quat qb = {curQ[b], curQ[nb + b], curQ[2*nb + b], curQ[3*nb + b]};
        float pb[3] = {curP[b], curP[nb + b], curP[2*nb + b]}, t[3];
        q_rot(qa, pb, t);
        Quat q = q_mul(qa, qb);
        if (r == R - 1) q = q_normalize(q);
        nxtP[b] = curP[a] + t[0]; nxtP[nb + b] = curP[nb + a] + t[1]; nxtP[2*nb + b] = curP[2*nb + a] + t[2];
        nxtQ[b] = q.w; nxtQ[nb + b] = q.x; nxtQ[2*nb + b] = q.y; nxtQ[3*nb + b] = q.z;
      }
      sync();
      float *tp = curP; curP = nxtP; nxtP = tp;
      float *tq = curQ; curQ = nxtQ; nxtQ = tq;
    }
    /* joint anchors and axes in the world frame */
    float *xanchor = s + m.L.xanchor, *xaxis = s + m.L.xaxis;
    for (int j = lane; j < nj; j += TEAM) {
      int b = MI(jnt_body, j);
      float anchor[3] = {mainP[b], mainP[nb + b], mainP[2*nb + b]}, axis[3] = {0.f, 0.f, 1.f};
      if (MI(jnt_type, j) != FB_JNT_FREE) {
        Quat q = {mainQ[b], mainQ[nb + b], mainQ[2*nb + b], mainQ[3*nb + b]};
        float jp[3] = {MF(jnt_pos, 3*j), MF(jnt_pos, 3*j+1), MF(jnt_pos, 3*j+2)};
        float ja[3] = {MF(jnt_axis, 3*j), MF(jnt_axis, 3*j+1), MF(jnt_axis, 3*j+2)}, t[3];
        q_rot(q, jp, t);
        anchor[0] += t[0]; anchor[1] += t[1]; anchor[2] += t[2];
        q_rot(q, ja, axis);
      }
      xanchor[j] = anchor[0]; xanchor[nj + j] = anchor[1]; xanchor[2*nj + j] = anchor[2];
      xaxis[j] = axis[0]; xaxis[nj + j] = axis[1]; xaxis[2*nj + j] = axis[2];
    }
    sync();
  }

  FB_MEM Quat body_quat(int b) const {
    const float *xquat = s + m.L.xquat;
    const int nb = m.nbody;
    Quat q = {xquat[b], xquat[nb + b], xquat[2*nb + b], xquat[3*nb + b]};
    return q;
  }

  /* ------------------------------------- A.2 xipos, com, cinert, cdof */
  FB_MEM void com_pos() {
    const int nb = m.nbody, nj = m.njnt, nv = m.nv;
    float *xpos = s + m.L.xpos, *xipos = s + m.L.xipos, *cin = s + m.L.cinert;
    float sx = 0.f, sy = 0.f, sz = 0.f;
    for (int b = 1 + lane; b < nb; b += TEAM) {
      float R[9], t[3];
      q_mat(body_quat(b), R);
      m_rot(R, MF(body_ipos, 3*b), MF(body_ipos, 3*b+1), MF(body_ipos, 3*b+2), t);
      float x = xpos[b] + t[0], y = xpos[nb + b] + t[1], z = xpos[2*nb + b] + t[2];
      xipos[b] = x; xipos[nb + b] = y; xipos[2*nb + b] = z;
      float mb = MF(body_mass, b);
      sx += mb*x; sy += mb*y; sz += mb*z;
    }
    sx = T::sum(mask, sx); sy = T::sum(mask, sy); sz = T::sum(mask, sz);
    sync();
    if (m.inv_total_mass > 0.f) {
      comx = sx*m.inv_total_mass; comy = sy*m.inv_total_mass; comz = sz*m.inv_total_mass;
    } else {
      comx = xipos[1]; comy = xipos[nb + 1]; comz = xipos[2*nb + 1];
    }
    for (int b = 1 + lane; b < nb; b += TEAM) {
      Quat bi = {MF(body_iquat, 4*b), MF(body_iquat, 4*b+1), MF(body_iquat, 4*b+2),
                 MF(body_iquat, 4*b+3)};
      float M[9];
      q_mat(q_mul(body_quat(b), bi), M);
      float i0 = MF(body_inertia, 3*b), i1 = MF(body_inertia, 3*b+1), i2 = MF(body_inertia, 3*b+2);
      float mb = MF(body_mass, b);
      float dx = xipos[b] - comx, dy = xipos[nb + b] - comy, dz = xipos[2*nb + b] - comz;
      cin[0*nb + b] = M[0]*M[0]*i0 + M[1]*M[1]*i1 + M[2]*M[2]*i2 + mb*(dy*dy + dz*dz);
      cin[1*nb + b] = M[3]*M[3]*i0 + M[4]*M[4]*i1 + M[5]*M[5]*i2 + mb*(dx*dx + dz*dz);
      cin[2*nb + b] = M[6]*M[6]*i0 + M[7]*M[7]*i1 + M[8]*M[8]*i2 + mb*(dx*dx + dy*dy);
      cin[3*nb + b] = M[0]*M[3]*i0 + M[1]*M[4]*i1 + M[2]*M[5]*i2 - mb*dx*dy;
      cin[4*nb + b] = M[0]*M[6]*i0 + M[1]*M[7]*i1 + M[2]*M[8]*i2 - mb*dx*dz;
      cin[5*nb + b] = M[3]*M[6]*i0 + M[4]*M[7]*i1 + M[5]*M[8]*i2 - mb*dy*dz;
      cin[6*nb + b] = mb*dx; cin[7*nb + b] = mb*dy; cin[8*nb + b] = mb*dz; cin[9*nb + b] = mb;
    }
    /* cdof about com, world axes */
    float *cdof = s + m.L.cdof;
    const float *xanchor = s + m.L.xanchor, *xaxis = s + m.L.xaxis;
    for (int j = lane; j < nj; j += TEAM) {
      int da = MI(jnt_dofadr, j), jtype = MI(jnt_type, j);
      float off[3] = {comx - xanchor[j], comy - xanchor[nj + j], comz - xanchor[2*nj + j]};
      if (jtype == FB_JNT_FREE) {
        float R[9];
        q_mat(body_quat(MI(jnt_body, j)), R);
        for (int i = 0; i < 3; i++) {
          for (int k = 0; k < 6; k++) cdof[k*nv + da + i] = (k == 3 + i) ? 1.f : 0.f;
          float ax[3] = {R[i], R[3 + i], R[6 + i]}, cr[3];
          v_cross(ax, off, cr);
          int d = da + 3 + i;
          cdof[d] = ax[0]; cdof[nv + d] = ax[1]; cdof[2*nv + d] = ax[2];
          cdof[3*nv + d] = cr[0]; cdof[4*nv + d] = cr[1]; cdof[5*nv + d] = cr[2];
        }
      } else {
        float ax[3] = {xaxis[j], xaxis[nj + j], xaxis[2*nj + j]};
        if (jtype == FB_JNT_HINGE) {
          float cr[3];
          v_cross(ax, off, cr);
          cdof[da] = ax[0]; cdof[nv + da] = ax[1]; cdof[2*nv + da] = ax[2];
          cdof[3*nv + da] = cr[0]; cdof[4*nv + da] = cr[1]; cdof[5*nv + da] = cr[2];
        } else {
          cdof[da] = 0.f; cdof[nv + da] = 0.f; cdof[2*nv + da] = 0.f;
          cdof[3*nv + da] = ax[0]; cdof[4*nv + da] = ax[1]; cdof[5*nv + da] = ax[2];
        }
      }
    }
    sync();
  }

  /* ---------------- A.4 comVel + the forward half of RNE (cacc) */
  /* cdof are all expressed about one point in world axes, so cvel[b] is the plain sum
   * of cdof*qvel over b's ancestor dofs and cacc[b] - cacc[world] the sum of
   * cdof_dot*qvel: two ancestor prefix sums by pointer jumping. */
  FB_MEM void prefix_sum6(float *mainb, float *altb) {
    const int nb = m.nbody, R = m.nround_anc;
    float *cur = (R & 1) ? altb : mainb, *nxt = (R & 1) ? mainb : altb;
    for (int r = 0; r < R; r++) {
      for (int b = lane; b < nb; b += TEAM) {
        int a = MI(body_anc, r*nb + b);
        for (int k = 0; k < 6; k++) nxt[k*nb + b] = cur[k*nb + b] + cur[k*nb + a];
      }
      sync();
      float *t = cur; cur = nxt; nxt = t;
    }
  }

  FB_MEM void com_vel_acc() {
    const int nb = m.nbody, nv = m.nv, R = m.nround_anc;
    const float *cdof = s + m.L.cdof, *qvel = s + m.L.qvel;
    float *cvel = s + m.L.cvel, *cacc = s + m.L.cacc;
    float *valt = s + m.L.cfrc, *aalt = s + m.L.crb;
    float *v0 = (R & 1) ? valt : cvel;
    for (int b = lane; b < nb; b += TEAM) {
      float v[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (b > 0) {
        int da = MI(body_dofadr, b), dn = MI(body_dofnum, b);
        for (int i = 0; i < dn; i++) {
          float qv = qvel[da + i];
          for (int k = 0; k < 6; k++) v[k] += cdof[k*nv + da + i]*qv;
        }
      }
      for (int k = 0; k < 6; k++) v0[k*nb + b] = v[k];
    }
    sync();
    prefix_sum6(cvel, valt);
    float *a0 = (R & 1) ? aalt : cacc;
    for (int b = lane; b < nb; b += TEAM) {
      float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      int jid = b > 0 ? MI(body_jnt, b) : -1;
      if (jid >= 0) {
        int p = MI(body_parent, b), da = MI(jnt_dofadr, jid);
        float cv[6];
        for (int k = 0; k < 6; k++) cv[k] = cvel[k*nb + p];
        if (MI(jnt_type, jid) == FB_JNT_FREE) {
          for (int i = 0; i < 3; i++) {         /* translations: cdof_dot = 0 */
            float qv = qvel[da + i];
            for (int k = 0; k < 6; k++) cv[k] += cdof[k*nv + da + i]*qv;
          }
          for (int i = 3; i < 6; i++) {         /* all three use cv after the translations */
            float cd[6], dd[6], qv = qvel[da + i];
            for (int k = 0; k < 6; k++) cd[k] = cdof[k*nv + da + i];
            cross_motion(cv, cd, dd);
            for (int k = 0; k < 6; k++) acc[k] += dd[k]*qv;
          }
        } else {
          float cd[6], dd[6], qv = qvel[da];
          for (int k = 0; k < 6; k++) cd[k] = cdof[k*nv + da];
          cross_motion(cv, cd, dd);
          for (int k = 0; k < 6; k++) acc[k] = dd[k]*qv;
        }
      }
      for (int k = 0; k < 6; k++) a0[k*nb + b] = acc[k];
    }
    sync();
    prefix_sum6(cacc, aalt);   /* cacc[world] = [0; -gravity] is added by the consumer */
  }

  /* --- per-body bias wrench minus applied wrench; composite inertia and wrench of
   * every subtree.  Bodies are in depth-first preorder, so a subtree is the id range
   * [b, b + size): its sum is assembled from power-of-two windows W_r[i] = sum of
   * 2^r consecutive bodies (doubling), following the bits of `size`.  No subtraction
   * of large prefixes, every lane busy, fixed summation order. */
  FB_MEM void body_forces_and_crb() {
    const int nb = m.nbody, R2 = m.nround_sub;
    const float *cin = s + m.L.cinert, *cvel = s + m.L.cvel, *cacc = s + m.L.cacc;
    const float *xipos = s + m.L.xipos, *xf = s + m.L.xfrc;
    float *A = s + m.L.crb, *B = s + m.L.altB;   /* 16 components x nb: crb | cfrc */
    float own[BPL][16];
FB_UNROLL
    for (int slot = 0; slot < BPL; slot++) {
      int b = lane + slot*TEAM;
      if (b >= nb) continue;
      float I[10], v[6], a[6], t0[6], t1[6], t2[6];
      for (int k = 0; k < 10; k++) I[k] = cin[k*nb + b];
      for (int k = 0; k < 6; k++) { v[k] = cvel[k*nb + b]; a[k] = cacc[k*nb + b]; }
      a[3] -= m.grav[0]; a[4] -= m.grav[1]; a[5] -= m.grav[2];
      inert_vec(I, a, t0);
      inert_vec(I, v, t1);
      cross_force(v, t1, t2);
      /* xfrc_applied: world force F, torque T at xipos -> spatial force about com */
      float F[3] = {xf[b], xf[nb + b], xf[2*nb + b]};
      float Tq[3] = {xf[3*nb + b], xf[4*nb + b], xf[5*nb + b]};
      float off[3] = {xipos[b] - comx, xipos[nb + b] - comy, xipos[2*nb + b] - comz}, cr[3];
      v_cross(off, F, cr);
      for (int k = 0; k < 10; k++) own[slot][k] = I[k];
      for (int k = 0; k < 3; k++) {
        own[slot][10 + k] = b > 0 ? t0[k] + t2[k] - (Tq[k] + cr[k]) : 0.f;
        own[slot][13 + k] = b > 0 ? t0[3+k] + t2[3+k] - F[k] : 0.f;
      }
    }
    sync();   /* cacc (aliases B) has been consumed by every lane */
FB_UNROLL
    for (int slot = 0; slot < BPL; slot++) {
      int b = lane + slot*TEAM;
      if (b >= nb) continue;
      for (int k = 0; k < 16; k++) A[k*nb + b] = own[slot][k];
    }
    sync();
    float acc[BPL][16];
    int pos[BPL], size[BPL];
FB_UNROLL
    for (int slot = 0; slot < BPL; slot++) {
      int b = lane + slot*TEAM;
      pos[slot] = b;
      size[slot] = b < nb ? MI(body_size, b) : 0;
      for (int k = 0; k < 16; k++) acc[slot][k] = 0.f;
    }
    float *cur = A, *nxt = B;
    for (int r = 0; r < R2; r++) {
      const int w = 1 << r;
FB_UNROLL
      for (int slot = 0; slot < BPL; slot++) {
        int b = lane + slot*TEAM;
        if (b >= nb) continue;
        if ((size[slot] >> r) & 1) {
          int p = pos[slot];
          for (int k = 0; k < 16; k++) acc[slot][k] += cur[k*nb + p];
          pos[slot] = p + w;
        }
        if (r + 1 < R2) {
          if (b + w < nb) for (int k = 0; k < 16; k++) nxt[k*nb + b] = cur[k*nb + b] + cur[k*nb + b + w];
          else for (int k = 0; k < 16; k++) nxt[k*nb + b] = cur[k*nb + b];
        }
      }
      sync();
      float *t = cur; cur = nxt; nxt = t;
    }
FB_UNROLL
    for (int slot = 0; slot < BPL; slot++) {
      int b = lane + slot*TEAM;
      if (b >= nb) continue;
      for (int k = 0; k < 16; k++) A[k*nb + b] = acc[slot][k];
    }
    sync();
  }

  /* ----------- A.3 mass matrix entries, bias, actuation, passive -> fsm */
  FB_MEM void mass_matrix_and_smooth() {
    const int nb = m.nbody, nv = m.nv, nu = m.nu;
    const float *crb = s + m.L.crb, *cfrc = s + m.L.cfrc, *cdof = s + m.L.cdof;
    const float *qpos = s + m.L.qpos, *qvel = s + m.L.qvel, *ctrl = s + m.L.ctrl;
    float *buf = s + m.L.buf, *fsm = s + m.L.fsm, *qM = s + m.L.qM, *actf = s + m.L.actf;
    for (int d = lane; d < nv; d += TEAM) {
      int b = MI(dof_body, d);
      float I[10], c[6], r[6], bias = 0.f;
      for (int k = 0; k < 10; k++) I[k] = crb[k*nb + b];
      for (int k = 0; k < 6; k++) { c[k] = cdof[k*nv + d]; bias += c[k]*cfrc[k*nb + b]; }
      inert_vec(I, c, r);
      for (int k = 0; k < 6; k++) buf[k*nv + d] = r[k];
      fsm[d] = -bias;
    }
    for (int a = lane; a < nu; a += TEAM) {
      int j = MI(act_jnt, a);
      float gear = MF(act_gear, a);
      float len = gear*qpos[MI(jnt_qposadr, j)], vel = gear*qvel[MI(jnt_dofadr, j)];
      float c = ctrl[a];
      if (MI(act_ctrllimited, a)) c = fminf(MF(act_ctrlrange, 2*a+1), fmaxf(MF(act_ctrlrange, 2*a), c));
      float f = MF(act_gain, a)*c + MF(act_bias, 3*a) + MF(act_bias, 3*a+1)*len + MF(act_bias, 3*a+2)*vel;
      if (MI(act_forcelimited, a)) f = fminf(MF(act_forcerange, 2*a+1), fmaxf(MF(act_forcerange, 2*a), f));
      actf[a] = f;
    }
    sync();
    for (int e = lane; e < m.nM; e += TEAM) {
      int i = MI(ent_i, e), j = MI(ent_j, e);
      float v = 0.f;
      for (int k = 0; k < 6; k++) v += cdof[k*nv + j]*buf[k*nv + i];
      if (i == j) v += MF(dof_armature, i);
      qM[e] = v;
    }
    for (int d = lane; d < nv; d += TEAM) {
      int j = MI(dof_jnt, d);
      float f = fsm[d];
      if (MI(jnt_type, j) != FB_JNT_FREE) {
        int qa = MI(jnt_qposadr, j);
        float stiff = g.ep_stiffness ? g.ep_stiffness[j*g.ep_pad] : MF(jnt_stiffness, j);
        if (stiff != 0.f) f -= stiff*(qpos[qa] - g.qpos_spring[qa]);
        int a0 = MI(jnt_actstart, j), a1 = MI(jnt_actstart, j + 1);
        for (int t = a0; t < a1; t++) { int a = MI(act_sorted, t); f += MF(act_gear, a)*actf[a]; }
      }
      f -= (g.ep_damping ? g.ep_damping[d*g.ep_pad] : MF(dof_damping, d))*qvel[d];
      fsm[d] = f;
    }
    sync();
  }

  /* ------------- scheduled sparse L'DL (mj_factorI) and solve (mj_solveLD) */
  /* qLD keeps the UNSCALED rows (U_ks = M_ks after elimination of k's descendants) and
   * dinv the inverse pivots, L_ks = U_ks*dinv[k]; the stage/lane schedule comes from
   * fb_build_model (deepest pivots first, one lane per destination word). */
  FB_MEM void factor(float hdamp) {
    const float *qM = s + m.L.qM;
    float *qLD = s + m.L.qLD;
    for (int e = lane; e < m.nM; e += TEAM) {
      int i = MI(ent_i, e);
      float v = qM[e];
      if (hdamp != 0.f && i == MI(ent_j, e)) v += hdamp*(g.ep_damping ? g.ep_damping[i*g.ep_pad] : MF(dof_damping, i));
      qLD[e] = v;
    }
    sync();
    eliminate();
  }

  /* in-place scheduled L'DL of the tree-sparse matrix held in qLD */
  FB_MEM void eliminate() {
    float *qLD = s + m.L.qLD, *dinv = s + m.L.dinv;
    const int NS = m.nstage;
    for (int st = 0; st < NS; st++) {
      int p0 = MI(st_pivstart, st), p1 = MI(st_pivstart, st + 1);
      for (int i = p0 + lane; i < p1; i += TEAM) {
        int k = MI(st_piv, i);
        dinv[k] = 1.0f/qLD[MI(dof_Madr, k)];
      }
      sync();
      int o0 = MI(fop_start, st*TEAM + lane), o1 = MI(fop_start, st*TEAM + lane + 1);
      for (int o = o0; o < o1; o++) {
        unsigned w0 = (unsigned)MI(fop, 2*o), w1 = (unsigned)MI(fop, 2*o + 1);
        qLD[w0 & 0xffffu] -= qLD[w0 >> 16]*dinv[w1 >> 16]*qLD[w1 & 0xffffu];
      }
      sync();
    }
  }

  /* x <- inv(L'DL) x, x in shared memory */
  FB_MEM void solve_ld(float *x) { solve_ld(x, s + m.L.tmp1); }
  FB_MEM void solve_ld(float *x, float *y) {
    const float *qLD = s + m.L.qLD, *dinv = s + m.L.dinv;
    const int NS = m.nstage;
    /* y = D^-1 L^-T x: leaves to root */
    for (int st = 0; st < NS; st++) {
      int p0 = MI(st_pivstart, st), p1 = MI(st_pivstart, st + 1);
      for (int i = p0 + lane; i < p1; i += TEAM) {
        int k = MI(st_piv, i);
        y[k] = x[k]*dinv[k];
      }
      sync();
      int o0 = MI(sop_start, st*TEAM + lane), o1 = MI(sop_start, st*TEAM + lane + 1);
      for (int o = o0; o < o1; o++) {
        unsigned w0 = (unsigned)MI(sop, 2*o), w1 = (unsigned)MI(sop, 2*o + 1);
        x[w0 & 0xffffu] -= qLD[w0 >> 16]*y[w1 >> 16];
      }
      sync();
    }
    /* x = L^-1 y: root to leaves, each dof gathers its (final) ancestors */
    for (int st = NS - 1; st >= 0; st--) {
      int p0 = MI(st_pivstart, st), p1 = MI(st_pivstart, st + 1);
      for (int i = p0 + lane; i < p1; i += TEAM) {
        int k = MI(st_piv, i), nk = MI(dof_nanc, k), adr = MI(dof_Madr, k);
        float acc = 0.f;
        for (int sdx = 1; sdx < nk; sdx++) acc += qLD[adr + sdx]*x[MI(ent_j, adr + sdx)];
        x[k] = y[k] - dinv[k]*acc;
      }
      sync();
    }
  }

  /* ---------------------------------- A.6/A.7 constraint detection */
  FB_MEM void detect_constraints() {
    const int nb = m.nbody, nj = m.njnt;
    const float *qpos = s + m.L.qpos, *qvel = s + m.L.qvel, *xpos = s + m.L.xpos;
    float *limf = s + m.L.limf;
    float *aref = g.efc, *D = g.efc + m.maxefc;
    int *con_cand = si + m.L.con_cand;
    /* joint limits: candidate lc = 2*j + side_index (0 lower, 1 upper) */
    float cnt = 0.f;
    for (int j = lane; j < nj; j += TEAM) {
      limf[j] = 0.f;
      int limited = MI(jnt_limited, j) && MI(jnt_type, j) != FB_JNT_FREE;
      float value = limited ? qpos[MI(jnt_qposadr, j)] : 0.f;
      float margin = MF(jnt_margin, j);
      for (int sd = 0; sd < 2; sd++) {
        float side = sd ? 1.f : -1.f;
        float dist = side*(MF(jnt_range, 2*j + sd) - value);
        float d = 0.f, ar = 0.f;
        if (limited && dist < margin) {
          float sr[2] = {MF(jnt_solref, 2*j), MF(jnt_solref, 2*j+1)}, si5[5];
          for (int k = 0; k < 5; k++) si5[k] = MF(jnt_solimp, 5*j + k);
          int dof = MI(jnt_dofadr, j);
          float K, B, imp, R;
          fb_row_params(m.timestep, sr, si5, dist - margin, MF(dof_invw, dof), &K, &B, &imp, &R);
          d = 1.0f/R;
          ar = -B*(-side*qvel[dof]) - K*imp*(dist - margin);
          cnt += 1.f;
        }
        D[2*j + sd] = d;
        aref[2*j + sd] = ar;
      }
    }
    nlim = (int)(T::sum(mask, cnt) + 0.5f);
    /* plane vs sphere / capsule end; compact in candidate order */
    int n = 0, npair = 0, nhard = 0;
    for (int c0 = 0; c0 < m.ncand; c0 += TEAM) {
      int c = c0 + lane;
      int hit = 0;
      float dist = 0.f, centre[3] = {0.f, 0.f, 0.f}, nrm[3] = {0.f, 0.f, 1.f}, R[9], radius = 0.f;
      float sup[3] = {0.f, 0.f, 0.f};      /* contact point on the geom relative to `centre`, before the -dist/2 n shift */
      int b = 0;
      if (c < m.ncand) {
        b = MI(cand_body, c);
        q_mat(body_quat(b), R);
        float t[3];
        m_rot(R, MF(cand_lpos, 3*c), MF(cand_lpos, 3*c+1), MF(cand_lpos, 3*c+2), t);
        centre[0] = xpos[b] + t[0]; centre[1] = xpos[nb + b] + t[1]; centre[2] = xpos[2*nb + b] + t[2];
        nrm[0] = MF(cand_pn, 3*c); nrm[1] = MF(cand_pn, 3*c+1); nrm[2] = MF(cand_pn, 3*c+2);
        radius = MF(cand_radius, c);
        float cdist = centre[0]*nrm[0] + centre[1]*nrm[1] + centre[2]*nrm[2] - MF(cand_pd, c);
        dist = cdist - radius;
        if (MI(cand_iscapsule, c) == 9 || MI(cand_iscapsule, c) == 10) {
          /* explicit <pair>, sphere-sphere (mjc_SphereSphere): the other sphere (geom1) sits on body
           * cand_body1 at cand_pn, radius cand_pd; the normal runs from it to this one */
          const int b1 = MI(cand_body1, c);
          float R1[9], t1[3];
          q_mat(body_quat(b1), R1);
          m_rot(R1, nrm[0], nrm[1], nrm[2], t1);
          float d[3] = {centre[0] - (xpos[b1] + t1[0]), centre[1] - (xpos[nb + b1] + t1[1]), centre[2] - (xpos[2*nb + b1] + t1[2])};
          const float len = sqrtf(d[0]*d[0] + d[1]*d[1] + d[2]*d[2]);
          if (len < FB_MINVAL) { nrm[0] = 1.f; nrm[1] = 0.f; nrm[2] = 0.f; }
          else { nrm[0] = d[0]/len; nrm[1] = d[1]/len; nrm[2] = d[2]/len; }
          dist = len - MF(cand_pd, c) - radius;
        }
        sup[0] = -nrm[0]*radius; sup[1] = -nrm[1]*radius; sup[2] = -nrm[2]*radius;
        if (MI(cand_iscapsule, c) == 4) {
          /* ellipsoid (mjc_PlaneConvex): support point along -normal, R Rg (s o normalize(s o (R Rg)'(-n))) */
          const Quat gq = {MF(cand_gquat, 4*c), MF(cand_gquat, 4*c+1), MF(cand_gquat, 4*c+2), MF(cand_gquat, 4*c+3)};
          float Rg[9], nb_[3], nl[3], w[3], wb[3];
          q_mat(gq, Rg);
          m_rot_t(R, nrm[0], nrm[1], nrm[2], nb_);
          m_rot_t(Rg, nb_[0], nb_[1], nb_[2], nl);
          for (int k = 0; k < 3; k++) w[k] = -nl[k]*MF(cand_laxis, 3*c+k);
          v_normalize3(w);
          for (int k = 0; k < 3; k++) w[k] *= MF(cand_laxis, 3*c+k);
          m_rot(Rg, w[0], w[1], w[2], wb);
          m_rot(R, wb[0], wb[1], wb[2], sup);
          dist = cdist + sup[0]*nrm[0] + sup[1]*nrm[1] + sup[2]*nrm[2];
        }
        if (MI(cand_iscapsule, c) >= 5 && MI(cand_iscapsule, c) <= 8) {
          /* cylinder point (mjc_PlaneCylinder) */
          const Quat gq = {MF(cand_gquat, 4*c), MF(cand_gquat, 4*c+1), MF(cand_gquat, 4*c+2), MF(cand_gquat, 4*c+3)};
          float Rg[9], axis[3], xaxis[3];
          q_mat(gq, Rg);
          m_rot(R, Rg[2], Rg[5], Rg[8], axis);
          m_rot(R, Rg[0], Rg[3], Rg[6], xaxis);
          dist = fb_plane_cylinder_point(nrm, axis, xaxis, MF(cand_laxis, 3*c), MF(cand_laxis, 3*c+1),
                                         MI(cand_iscapsule, c) - 5, cdist, sup);
        }
        hit = dist < MF(cand_margin, c) - MF(cand_gap, c);
        if ((MI(cand_iscapsule, c) & ~1) == 2) {
          /* box corner (mjc_PlaneBox): only while it is below the box centre along the normal.
           * (MuJoCo's cap of 4 corners per box only binds in degenerate poses and is not applied
           * here; the per-thread kernel and the oracle apply it.) */
          float u[3];
          m_rot(R, MF(cand_lpos, 3*c) - MF(cand_laxis, 3*c), MF(cand_lpos, 3*c+1) - MF(cand_laxis, 3*c+1),
                MF(cand_lpos, 3*c+2) - MF(cand_laxis, 3*c+2), u);
          if (u[0]*nrm[0] + u[1]*nrm[1] + u[2]*nrm[2] > 0.f) hit = 0;
        }
      }
      unsigned bits = T::ballot(mask, base, hit);
      npair += FB_POPC(T::ballot(mask, base, hit && MI(cand_iscapsule, c) == 9));
      if (m.n_hard > 0) nhard += FB_POPC(T::ballot(mask, base, hit && MI(cand_iscapsule, c) == 10));
      if (hit) {
        int i = n + FB_POPC(bits & ((1u << lane) - 1u));
        con_cand[i] = c;
        g.d_con_cand[i] = c;
        g.d_con_dist[i] = dist;
        float f[9];
        for (int k = 0; k < 3; k++) {
          g.d_con_pos[3*i + k] = MI(cand_iscapsule, c) >= 4 ? centre[k] + sup[k] - nrm[k]*0.5f*dist
                                                            : centre[k] - nrm[k]*(radius + 0.5f*dist);
          f[k] = nrm[k];
        }
        if (MI(cand_iscapsule, c) == 1) {
          m_rot(R, MF(cand_laxis, 3*c), MF(cand_laxis, 3*c+1), MF(cand_laxis, 3*c+2), f + 3);
        } else {
          f[3] = f[4] = f[5] = 0.f;
        }
        /* mju_makeFrame */
        v_normalize3(f);
        if (sqrtf(f[3]*f[3] + f[4]*f[4] + f[5]*f[5]) < 0.5f) {
          f[3] = f[4] = f[5] = 0.f;
          if (f[1] < 0.5f && f[1] > -0.5f) f[4] = 1.f; else f[5] = 1.f;
        }
        float dt = f[0]*f[3] + f[1]*f[4] + f[2]*f[5];
        f[3] -= dt*f[0]; f[4] -= dt*f[1]; f[5] -= dt*f[2];
        v_normalize3(f + 3);
        v_cross(f, f + 3, f + 6);
        for (int k = 0; k < 9; k++) g.d_con_frame[9*i + k] = f[k];
      }
      n += FB_POPC(bits);
    }
    ncon = n;
    npair_act = npair;
    nhard_act = nhard;
    if (lane == 0) *g.d_ncon = n;
    sync();
  }

  /* ---------------------------- contact rows: J3, D, aref (A.7) */
  FB_MEM void make_contact_rows() {
    const int nv = m.nv, nj = m.njnt;
    const float *cdof = s + m.L.cdof, *qvel = s + m.L.qvel;
    const int *con_cand = si + m.L.con_cand;
    float *aref = g.efc, *D = g.efc + m.maxefc;
    for (int i = 0; i < ncon; i++) {
      int c = con_cand[i], b = MI(cand_body, c), b1 = MI(cand_body1, c);
      float off[3] = {g.d_con_pos[3*i] - comx, g.d_con_pos[3*i+1] - comy, g.d_con_pos[3*i+2] - comz};
      float f[9];
      for (int k = 0; k < 9; k++) f[k] = g.d_con_frame[9*i + k];
      for (int v = lane; v < nv; v += TEAM) {
        float j0 = 0.f, j1 = 0.f, j2 = 0.f;
        /* mj_jacDifPair: the point's velocity on geom2's body minus the one on geom1's (the world for
         * plane candidates); dofs above both bodies cancel */
        const int in2 = (int)((unsigned)MI(body_ancmask, b*m.nmaskw + (v >> 5)) >> (v & 31) & 1u);
        const int in1 = b1 > 0 ? (int)((unsigned)MI(body_ancmask, b1*m.nmaskw + (v >> 5)) >> (v & 31) & 1u) : 0;
        if (in2 != in1) {
          float ang[3] = {cdof[v], cdof[nv + v], cdof[2*nv + v]}, cr[3];
          v_cross(ang, off, cr);
          const float sg = in2 ? 1.f : -1.f;
          float lx = sg*(cdof[3*nv + v] + cr[0]), ly = sg*(cdof[4*nv + v] + cr[1]), lz = sg*(cdof[5*nv + v] + cr[2]);
          j0 = f[0]*lx + f[1]*ly + f[2]*lz;
          j1 = f[3]*lx + f[4]*ly + f[5]*lz;
          j2 = f[6]*lx + f[7]*ly + f[8]*lz;
        }
        g.J3[(3*i)*nv + v] = j0; g.J3[(3*i+1)*nv + v] = j1; g.J3[(3*i+2)*nv + v] = j2;
      }
    }
    sync();
    j3_times(qvel);  /* prod3 <- J3 qvel */
    for (int i = lane; i < ncon; i += TEAM) {
      int c = con_cand[i];
      float mu = cand_mu(c), dist = g.d_con_dist[i];
      float includemargin = MF(cand_margin, c) - MF(cand_gap, c);
      float sr[2] = {MF(cand_solref, 2*c), MF(cand_solref, 2*c+1)}, si5[5];
      for (int k = 0; k < 5; k++) si5[k] = MF(cand_solimp, 5*c + k);
      float tran = MF(cand_invw, c);
      float K, B, imp, R;
      fb_row_params(m.timestep, sr, si5, dist - includemargin, tran + mu*mu*tran, &K, &B, &imp, &R);
      float impratio = fmaxf(FB_MINVAL, m.impratio);
      float R1 = R/impratio;
      float cmu2 = mu*mu*(R1/R);
      float Rpy = fmaxf(FB_MINVAL, 2.f*cmu2*R1);
      float vn = g.prod3[3*i], vt1 = g.prod3[3*i+1], vt2 = g.prod3[3*i+2];
      if (MI(cand_iscapsule, c) == 10) {
        /* frictionless pair: one hard row Jn a >= aref_n with a multiplier (solve_constraints).  Its
         * four slots carry D = 0 -- the soft rows' sums skip them -- and aref_n, the mean of the four
         * pyramidal aref (the +-mu vt terms cancel) */
        for (int sub = 0; sub < 4; sub++) {
          D[2*nj + 4*i + sub] = 0.f;
          aref[2*nj + 4*i + sub] = -B*vn - K*imp*(dist - includemargin);
        }
        continue;
      }
      for (int sub = 0; sub < 4; sub++) {
        float sg = (sub & 1) ? -1.f : 1.f;
        float vel = vn + sg*mu*((sub < 2) ? vt1 : vt2);
        int r = 2*nj + 4*i + sub;
        D[r] = 1.0f/Rpy;
        aref[r] = -B*vel - K*imp*(dist - includemargin);
      }
    }
    if (nhard_act > 0 && lane == 0) {
      int h = 0;
      for (int i = 0; i < ncon; i++) if (MI(cand_iscapsule, con_cand[i]) == 10) si[m.L.hcon + h++] = i;
    }
    sync();
  }

  /* prod3[r3] <- sum_v J3[r3][v] x[v] */
  FB_MEM void j3_times(const float *x) {
    const int nv = m.nv;
    for (int r3 = 0; r3 < 3*ncon; r3++) {
      float part = 0.f;
      for (int v = lane; v < nv; v += TEAM) part += g.J3[r3*nv + v]*x[v];
      part = T::sum(mask, part);
      if (lane == 0) g.prod3[r3] = part;
    }
    sync();
  }

  /* out[r] <- J_r x for every row (limit candidates, then contact rows) */
  FB_MEM void rows_apply(const float *x, float *out) {
    const int nj = m.njnt;
    j3_times(x);
    for (int j = lane; j < nj; j += TEAM) {
      float xv = x[MI(jnt_dofadr, j)];
      out[2*j] = xv;       /* lower: jac = +1 */
      out[2*j + 1] = -xv;  /* upper: jac = -1 */
    }
    const int *con_cand = si + m.L.con_cand;
    for (int i = lane; i < ncon; i += TEAM) {
      float mu = cand_mu(con_cand[i]);
      float pn = g.prod3[3*i], p1 = g.prod3[3*i+1], p2 = g.prod3[3*i+2];
      int r = 2*nj + 4*i;
      out[r] = pn + mu*p1; out[r+1] = pn - mu*p1; out[r+2] = pn + mu*p2; out[r+3] = pn - mu*p2;
    }
    sync();
  }

  /* out[v] (+)= sum_r J_r[v] y[r];  y in global efc scratch */
  FB_MEM void rows_tapply(const float *y, float *out, int accumulate) {
    const int nv = m.nv, nj = m.njnt;
    const int *con_cand = si + m.L.con_cand;
    float *y3 = g.prod3 + 3*m.maxcon;
    for (int i = lane; i < ncon; i += TEAM) {
      float mu = cand_mu(con_cand[i]);
      const float *yy = y + 2*nj + 4*i;
      y3[3*i] = yy[0] + yy[1] + yy[2] + yy[3];
      y3[3*i+1] = mu*(yy[0] - yy[1]);
      y3[3*i+2] = mu*(yy[2] - yy[3]);
    }
    sync();
    for (int v = lane; v < nv; v += TEAM) {
      float acc = accumulate ? out[v] : 0.f;
      int j = MI(dof_jnt, v);
      if (MI(jnt_type, j) != FB_JNT_FREE) acc += y[2*j] - y[2*j + 1];
      for (int r3 = 0; r3 < 3*ncon; r3++) acc += g.J3[r3*nv + v]*y3[r3];
      out[v] = acc;
    }
    sync();
  }

  /* out = M x on the tree-sparse layout: ancestors from the dof's own row, descendants from
   * the column lists */
  FB_MEM void mul_m(const float *x, float *out) {
    const int nv = m.nv;
    const float *qM = s + m.L.qM;
    for (int i = lane; i < nv; i += TEAM) {
      const int adr = MI(dof_Madr, i), nk = MI(dof_nanc, i);
      float acc = 0.f;
      for (int k = 0; k < nk; k++) acc += qM[adr + k]*x[MI(ent_j, adr + k)];
      for (int t = MI(col_start, i); t < MI(col_start, i + 1); t++) acc += qM[MI(col_ent, t)]*x[MI(col_dof, t)];
      out[i] = acc;
    }
    sync();
  }

  /* x <- H^-1 x with the dense Cholesky factor held in L.H (lower triangle): L y = x, L' x = y */
  FB_MEM void dense_solve(float *x) {
    const int nv = m.nv;
    const float *H = s + m.L.H;
    for (int k = 0; k < nv; k++) {
      const float yk = x[k]/H[k*nv + k];
      sync();
      if (lane == 0) x[k] = yk;
      for (int i = k + 1 + lane; i < nv; i += TEAM) x[i] -= H[i*nv + k]*yk;
      sync();
    }
    for (int k = nv - 1; k >= 0; k--) {
      const float xk = x[k]/H[k*nv + k];
      sync();
      if (lane == 0) x[k] = xk;
      for (int i = lane; i < k; i += TEAM) x[i] -= H[k*nv + i]*xk;
      sync();
    }
  }

  /* ---------- hard normal rows of frictionless pairs (kind 10): equality-constrained Newton ----------
   * Each active hard contact h (contact hcon[h]) has one row Jn_h = J3[3 i] with Jn_h a >= aref_h and a
   * multiplier lambda_h >= 0, its normal force.  On the working set W (hon[h] = 1; -1: a row that
   * depends on the others of W, out for the rest of the solve, force 0) the Newton step is
   * taken in direct-multiplier form: u = H^-1 g, V = H^-1 Jn_W', S = Jn_W V, S lambda = Jn_W u - x_W,
   * p = -u + V lambda, so that Jn_W (a + p) = aref_W.  A row counts as satisfied while
   * |Jn a - aref| <= FB_HARD_TOL (sum_v |Jn_v a_v| + |aref| + S_hh |lambda_h|) + FB_HARD_ATOL: relative to
   * the terms the residual is the difference of and to the normal acceleration its own force makes --
   * one ulp of lambda moves Jn a by S_hh ulp(lambda), the floor a Newton step cannot go below. */
#define FB_HARD_TOL 1e-4f
#define FB_HARD_ATOL 1e-6f
#define FB_HARD_PIVOT 1e-5f    /* a pivot of S below this share of its diagonal: the row depends on the others */
/* On a settled W the Lagrangian gradient can stay above the soft solver's 2e-5 floor: the stiff soft
 * rows (joint limits) put rounding noise of D eps |J a| into it, and the Newton steps it drives are
 * ~1e-5 of |qacc| (SALAMANDER, both foot pairs and a joint limit active).  A step below 1e-4 of |qacc|
 * on a settled W therefore counts as converged too. */
#define FB_HARD_STALL 1e-8f

  /* hx = Jn a - aref and its tolerance for every active hard row; prod3 holds J3 a */
  FB_MEM void hard_residuals(const float *a) {
    const int nv = m.nv, nj = m.njnt, NH = m.n_hard;
    const int *hcon = si + m.L.hcon;
    float *hx = s + m.L.hx, *htol = s + m.L.htol;
    const float *S = s + m.L.hS, *hlam = s + m.L.hlam;
    for (int h = 0; h < nhard_act; h++) {
      const int i = hcon[h];
      float mag = 0.f;
      for (int v = lane; v < nv; v += TEAM) mag += fabsf(g.J3[(3*i)*nv + v]*a[v]);
      mag = T::sum(mask, mag);
      if (lane == 0) {
        const float ar = g.efc[2*nj + 4*i];
        /* (a non-zero multiplier was computed together with its S_hh) */
        const float own = hlam[h] != 0.f ? S[h*NH + h]*fabsf(hlam[h]) : 0.f;
        hx[h] = g.prod3[3*i] - ar;
        htol[h] = FB_HARD_TOL*(mag + fabsf(ar) + own) + FB_HARD_ATOL;
      }
    }
    sync();
  }

  /* violated rows outside W join it; returns whether any did (the same on every lane) */
  FB_MEM int hard_add_violated() {
    int *hon = si + m.L.hon;
    const float *hx = s + m.L.hx, *htol = s + m.L.htol;
    int add = 0;
    for (int h = 0; h < nhard_act; h++) add |= hon[h] == 0 && hx[h] < -htol[h];
    sync();
    if (lane == 0) for (int h = 0; h < nhard_act; h++) if (hon[h] == 0 && hx[h] < -htol[h]) hon[h] = 1;
    sync();
    return add;
  }

  FB_MEM int hard_feasible() {
    const int *hon = si + m.L.hon;
    const float *hx = s + m.L.hx, *htol = s + m.L.htol;
    for (int h = 0; h < nhard_act; h++) if (hon[h] == 1 && fabsf(hx[h]) > htol[h]) return 0;
    return 1;
  }

  /* the row of W with the most negative multiplier leaves W; returns whether there was one */
  FB_MEM int hard_release() {
    int *hon = si + m.L.hon;
    float *hlam = s + m.L.hlam;
    int worst = -1;
    for (int h = 0; h < nhard_act; h++)
      if (hon[h] == 1 && hlam[h] < 0.f && (worst < 0 || hlam[h] < hlam[worst])) worst = h;
    sync();
    if (lane == 0 && worst >= 0) { hon[worst] = 0; hlam[worst] = 0.f; }
    sync();
    return worst >= 0;
  }

  /* |g - Jn_W' lambda|^2, the gradient of the Lagrangian with the multipliers of the last step;
   * |Jn_W' lambda|^2 is added to *gref, the terms the gradient is the difference of */
  FB_MEM float hard_lagrangian_norm2(const float *grad, float *gref) {
    const int nv = m.nv;
    const int *hcon = si + m.L.hcon, *hon = si + m.L.hon;
    const float *hlam = s + m.L.hlam;
    float gn = 0.f, fn = 0.f;
    for (int v = lane; v < nv; v += TEAM) {
      float f = 0.f;
      for (int h = 0; h < nhard_act; h++) if (hon[h] == 1) f += hlam[h]*g.J3[(3*hcon[h])*nv + v];
      const float gl = grad[v] - f;
      gn += gl*gl; fn += f*f;
    }
    *gref += T::sum(mask, fn);
    return T::sum(mask, gn);
  }

  /* sum over W of lambda_h Jn_h p (prod3 holds J3 p): the hard rows' term of the Lagrangian's slope */
  FB_MEM float hard_lambda_jp() {
    const int *hcon = si + m.L.hcon, *hon = si + m.L.hon;
    const float *hlam = s + m.L.hlam;
    float acc = 0.f;
    for (int h = 0; h < nhard_act; h++) if (hon[h] == 1) acc += hlam[h]*g.prod3[3*hcon[h]];
    return acc;
  }

  /* p = -H^-1 g on entry (H factored: dense while a kind-9 pair is active, else tree-sparse in qLD);
   * on return p = -u + V lambda with the multipliers of W in hlam.  y: nv floats of scratch. */
  FB_MEM void hard_step(float *p, float *y) {
    const int nv = m.nv, NH = m.n_hard;
    const int *hcon = si + m.L.hcon;
    int *hon = si + m.L.hon, *ws = si + m.L.hws;
    float *V = s + m.L.hV, *S = s + m.L.hS, *Lf = s + m.L.hL, *hlam = s + m.L.hlam, *rhs = s + m.L.hrhs;
    const float *hx = s + m.L.hx;
    int any = 0;
    for (int h = 0; h < nhard_act; h++) {
      if (hon[h] != 1) continue;
      any = 1;
      const float *jn = g.J3 + (3*hcon[h])*nv;
      for (int v = lane; v < nv; v += TEAM) V[h*nv + v] = jn[v];
      sync();
      if (npair_act > 0) dense_solve(V + h*nv); else solve_ld(V + h*nv, y);
    }
    if (!any) return;
    for (int a = 0; a < nhard_act; a++) {
      if (hon[a] != 1) continue;
      const float *jn = g.J3 + (3*hcon[a])*nv;
      for (int b = 0; b <= a; b++) {
        if (hon[b] != 1) continue;
        float part = 0.f;
        for (int v = lane; v < nv; v += TEAM) part += jn[v]*V[b*nv + v];
        part = T::sum(mask, part);
        if (lane == 0) S[a*NH + b] = part;
      }
      float part = 0.f;                       /* Jn_a u = -Jn_a p */
      for (int v = lane; v < nv; v += TEAM) part -= jn[v]*p[v];
      part = T::sum(mask, part);
      if (lane == 0) rhs[a] = part - hx[a];
    }
    sync();
    if (lane == 0) {
      /* Cholesky of S on W (compact order ws); a row whose pivot collapses leaves W */
      for (;;) {
        int k = 0;
        for (int h = 0; h < nhard_act; h++) if (hon[h] == 1) ws[k++] = h;
        int drop = -1;
        for (int a = 0; a < k && drop < 0; a++) {
          for (int b = 0; b <= a; b++) {
            float sum = S[ws[a]*NH + ws[b]];
            for (int c = 0; c < b; c++) sum -= Lf[a*NH + c]*Lf[b*NH + c];
            if (b < a) { Lf[a*NH + b] = sum/Lf[b*NH + b]; continue; }
            if (!(sum > FB_HARD_PIVOT*S[ws[a]*NH + ws[a]])) { drop = ws[a]; break; }
            Lf[a*NH + a] = sqrtf(sum);
          }
        }
        if (drop >= 0) { hon[drop] = -1; hlam[drop] = 0.f; continue; }
        for (int a = 0; a < k; a++) {
          float sum = rhs[ws[a]];
          for (int c = 0; c < a; c++) sum -= Lf[a*NH + c]*hlam[ws[c]];
          hlam[ws[a]] = sum/Lf[a*NH + a];
        }
        for (int a = k - 1; a >= 0; a--) {
          float sum = hlam[ws[a]];
          for (int c = a + 1; c < k; c++) sum -= Lf[c*NH + a]*hlam[ws[c]];
          hlam[ws[a]] = sum/Lf[a*NH + a];
        }
        break;
      }
    }
    sync();
    for (int v = lane; v < nv; v += TEAM) {
      float acc = p[v];
      for (int h = 0; h < nhard_act; h++) if (hon[h] == 1) acc += hlam[h]*V[h*nv + v];
      p[v] = acc;
    }
    sync();
  }

  /* ratio test: alpha shrinks to where the first hard row outside W would become violated along p
   * (prod3 holds J3 p); returns that row (it joins W after the step) or -1 */
  FB_MEM int hard_ratio_test(float *alpha) {
    const int *hcon = si + m.L.hcon, *hon = si + m.L.hon;
    const float *hx = s + m.L.hx;
    int block = -1;
    for (int h = 0; h < nhard_act; h++) {
      if (hon[h] != 0) continue;
      const float jp = g.prod3[3*hcon[h]];
      if (!(jp < 0.f)) continue;
      const float ah = fmaxf(0.f, -hx[h]/jp);
      if (ah < *alpha) { *alpha = ah; block = h; }
    }
    return block;
  }

  /* ------------------------------------ A.8 primal Newton, exact line search */
  FB_MEM void solve_constraints(float *tmp1, float *tmp2) {
    const int nv = m.nv, nj = m.njnt;
    const int nrow = 2*nj + 4*ncon;
    const int *con_cand = si + m.L.con_cand;
    float *qacc = s + m.L.qacc, *fsm = s + m.L.fsm, *fcon = s + m.L.fcon;
    float *grad = s + m.L.grad, *p = s + m.L.pvec, *qLD = s + m.L.qLD;
    const float *qM = s + m.L.qM;
    float *aref = g.efc, *D = g.efc + m.maxefc, *res = g.efc + 2*m.maxefc,
          *jp = g.efc + 3*m.maxefc, *frc = g.efc + 4*m.maxefc;
    int maxit = m.solver_iterations < 50 ? m.solver_iterations : 50;
    /* hard rows of frictionless pairs: W starts empty; `done` once the multipliers of W are >= 0,
     * W's rows hold and no other row is violated */
    int done = 0;
    if (nhard_act > 0) {
      for (int h = lane; h < nhard_act; h += TEAM) { si[m.L.hon + h] = 0; s[m.L.hlam + h] = 0.f; }
      sync();
    }
    for (int it = 0; it < maxit; it++) {
      rows_apply(qacc, res);
      for (int r = lane; r < nrow; r += TEAM) {
        float rr = res[r] - aref[r];
        res[r] = rr;
        frc[r] = (rr < 0.f) ? D[r]*rr : 0.f;   /* y = D min(0, res) */
      }
      sync();
      if (nhard_act > 0) hard_residuals(qacc);   /* prod3 = J3 qacc */
      mul_m(qacc, tmp1);                         /* tmp1 = M a */
      float gref = 0.f;                          /* magnitude of the terms the gradient is the difference of */
      for (int v = lane; v < nv; v += TEAM) {
        gref += tmp1[v]*tmp1[v] + fsm[v]*fsm[v];
        tmp1[v] -= fsm[v]; grad[v] = tmp1[v];
      }
      gref = T::sum(mask, gref);
      sync();
      rows_tapply(frc, grad, 1);                 /* grad = M a - fsm + J' y */
      int added = 0, feasible = 1;
      if (nhard_act == 0) {
        float gn = 0.f;
        for (int v = lane; v < nv; v += TEAM) gn += grad[v]*grad[v];
        gn = T::sum(mask, gn);
        /* MuJoCo's test (scaled gradient < tolerance, 1e-8 by default) is out of reach of fp32:
         * once the active set is right the gradient is rounding noise, ~5e-6 of the terms it is
         * the difference of.  Stop at whichever floor comes first. */
        if (sqrtf(gn)*m.solver_scale < fmaxf(m.tolerance, 2e-5f*sqrtf(gref)*m.solver_scale)) break;
      } else {
        /* the same test on the Lagrangian gradient, once W is settled and its rows hold; then a
         * negative multiplier leaves W, or the solve is done */
        added = hard_add_violated();
        feasible = hard_feasible();
        const float gn = hard_lagrangian_norm2(grad, &gref);
        if (!added && feasible && sqrtf(gn)*m.solver_scale < fmaxf(m.tolerance, 2e-5f*sqrtf(gref)*m.solver_scale)) {
          if (!hard_release()) { done = 1; break; }
        }
      }
      /* H = M + sum_active D J'J.  Every row of J is supported on the ancestors of ONE body
       * (limits: one dof; plane contacts: the chain of the touching body), so H has exactly the
       * tree sparsity of M: it is assembled in M's layout and factored by the same scheduled
       * sparse L'DL (leaves first), no dense 33x33 matrix. */
      if (npair_act > 0) {
        /* A contact of an explicit <pair> is active: its rows live on the chains of two bodies, so
         * J'DJ couples dofs that are not ancestors of one another and H loses the tree sparsity.
         * Dense H (lower triangle) in the environment's shared memory, Cholesky in place, two
         * triangular solves. */
        float *H = s + m.L.H;
        for (int idx = lane; idx < nv*nv; idx += TEAM) H[idx] = 0.f;
        sync();
        for (int e = lane; e < m.nM; e += TEAM) {
          const int u = MI(ent_i, e), v = MI(ent_j, e);      /* v is u or an ancestor of u: v <= u */
          float h = qM[e];
          if (u == v) {
            int j = MI(dof_jnt, u);
            if (MI(jnt_type, j) != FB_JNT_FREE) {
              if (res[2*j] < 0.f) h += D[2*j];
              if (res[2*j+1] < 0.f) h += D[2*j+1];
            }
          }
          H[(u > v ? u : v)*nv + (u > v ? v : u)] = h;
        }
        sync();
        for (int idx = lane; idx < nv*nv; idx += TEAM) {
          const int u = idx/nv, v = idx - u*nv;
          if (v > u) continue;
          float h = H[idx];
          for (int i = 0; i < ncon; i++) {
            const int r = 2*nj + 4*i;
            const float d = D[r], mu = cand_mu(con_cand[i]);
            const float nu_ = g.J3[(3*i)*nv + u], nv_ = g.J3[(3*i)*nv + v];
            const float t1u = mu*g.J3[(3*i+1)*nv + u], t1v = mu*g.J3[(3*i+1)*nv + v];
            const float t2u = mu*g.J3[(3*i+2)*nv + u], t2v = mu*g.J3[(3*i+2)*nv + v];
            if (res[r] < 0.f) h += d*(nu_ + t1u)*(nv_ + t1v);
            if (res[r+1] < 0.f) h += d*(nu_ - t1u)*(nv_ - t1v);
            if (res[r+2] < 0.f) h += d*(nu_ + t2u)*(nv_ + t2v);
            if (res[r+3] < 0.f) h += d*(nu_ - t2u)*(nv_ - t2v);
          }
          H[idx] = h;
        }
        sync();
        for (int k = 0; k < nv; k++) {
          const float piv = sqrtf(H[k*nv + k]), inv = 1.0f/piv;
          for (int i = k + 1 + lane; i < nv; i += TEAM) H[i*nv + k] *= inv;
          sync();
          if (lane == 0) H[k*nv + k] = piv;
          for (int i = k + 1 + lane; i < nv; i += TEAM) {
            const float lik = H[i*nv + k];
            for (int j = k + 1; j <= i; j++) H[i*nv + j] -= lik*H[j*nv + k];
          }
          sync();
        }
        /* p = -H^-1 grad */
        for (int v = lane; v < nv; v += TEAM) p[v] = -grad[v];
        sync();
        dense_solve(p);
      } else {
        for (int e = lane; e < m.nM; e += TEAM) {
          const int u = MI(ent_i, e), v = MI(ent_j, e);      /* v is u or an ancestor of u */
          float h = qM[e];
          if (u == v) {
            int j = MI(dof_jnt, u);
            if (MI(jnt_type, j) != FB_JNT_FREE) {
              if (res[2*j] < 0.f) h += D[2*j];
              if (res[2*j+1] < 0.f) h += D[2*j+1];
            }
          }
          for (int i = 0; i < ncon; i++) {
            int c = con_cand[i], b = MI(cand_body, c);
            /* u on the chain of b implies v on it too */
            if (!(((unsigned)MI(body_ancmask, b*m.nmaskw + (u >> 5)) >> (u & 31)) & 1u)) continue;
            int r = 2*nj + 4*i;
            float d = D[r], mu = cand_mu(c);
            float nu_ = g.J3[(3*i)*nv + u], nv_ = g.J3[(3*i)*nv + v];
            float t1u = mu*g.J3[(3*i+1)*nv + u], t1v = mu*g.J3[(3*i+1)*nv + v];
            float t2u = mu*g.J3[(3*i+2)*nv + u], t2v = mu*g.J3[(3*i+2)*nv + v];
            if (res[r] < 0.f) h += d*(nu_ + t1u)*(nv_ + t1v);
            if (res[r+1] < 0.f) h += d*(nu_ - t1u)*(nv_ - t1v);
            if (res[r+2] < 0.f) h += d*(nu_ + t2u)*(nv_ + t2v);
            if (res[r+3] < 0.f) h += d*(nu_ - t2u)*(nv_ - t2v);
          }
          qLD[e] = h;
        }
        sync();
        eliminate();
        /* p = -H^-1 grad */
        for (int v = lane; v < nv; v += TEAM) p[v] = -grad[v];
        sync();
        solve_ld(p, tmp2);
      }
      if (nhard_act > 0) hard_step(p, tmp2);
      float alpha = 1.0f;
      if (nhard_act > 0 && (added || !feasible)) {
        /* W grew or its rows do not hold yet: the full step onto them */
        j3_times(p);
      } else {
        /* exact line search on phi'(alpha) = g0 + alpha pMp + sum D jp min(0, res + alpha jp).  With
         * hard rows it runs on the Lagrangian, lambda of W held: g0 loses lambda Jn_W p (Jn_W p =
         * -x_W, rounding noise once the rows hold, which would otherwise steer alpha) */
        rows_apply(p, jp);
        mul_m(p, tmp2);
        float pMp = 0.f, g0 = 0.f;
        for (int v = lane; v < nv; v += TEAM) { pMp += p[v]*tmp2[v]; g0 += p[v]*tmp1[v]; }
        pMp = T::sum(mask, pMp);
        g0 = T::sum(mask, g0);
        if (nhard_act > 0) g0 -= hard_lambda_jp();
        float lo = 0.f, hi = 3.0e38f;
        for (int r = lane; r < nrow; r += TEAM) {
          float dr = D[r], jr = jp[r];
          if (dr <= 0.f || jr == 0.f) continue;
          float al = -res[r]/jr;
          if (!(al > 0.f)) continue;
          float gv = g0 + al*pMp;
          for (int q = 0; q < nrow; q++) {
            float dq = D[q];
            if (dq > 0.f) gv += dq*jp[q]*fminf(0.f, res[q] + al*jp[q]);
          }
          if (gv <= 0.f) lo = fmaxf(lo, al); else hi = fminf(hi, al);
        }
        lo = T::max(mask, lo);
        hi = T::min(mask, hi);
        float am = hi < 1.0e38f ? 0.5f*(lo + hi) : lo + 1.0f;
        float glo = 0.f, slope = 0.f;
        for (int r = lane; r < nrow; r += TEAM) {
          float dr = D[r];
          if (dr <= 0.f) continue;
          float jr = jp[r];
          glo += dr*jr*fminf(0.f, res[r] + lo*jr);
          if (res[r] + am*jr < 0.f) slope += dr*jr*jr;
        }
        glo = T::sum(mask, glo) + g0 + lo*pMp;
        slope = T::sum(mask, slope) + pMp;
        alpha = slope > 0.f ? lo - glo/slope : 1.0f;
        if (!(alpha > 0.f) || alpha != alpha) alpha = lo > 0.f ? lo : 1.0f;
        if (hi < 1.0e38f && alpha > hi) alpha = hi;
      }
      const int block = nhard_act > 0 ? hard_ratio_test(&alpha) : -1;   /* prod3 = J3 p */
      float st = 0.f, a2 = 0.f;
      for (int v = lane; v < nv; v += TEAM) {
        float dv = alpha*p[v], nvv = qacc[v] + dv;
        st += dv*dv; a2 += nvv*nvv;
      }
      st = T::sum(mask, st);
      a2 = T::sum(mask, a2);
      sync();
      for (int v = lane; v < nv; v += TEAM) qacc[v] += alpha*p[v];
      if (block >= 0 && lane == 0) si[m.L.hon + block] = 1;
      sync();
      if (nhard_act == 0) {
        if (st <= 1e-14f*a2) break;
      } else if (st <= FB_HARD_STALL*a2 && !added && feasible && block < 0) {
        /* a vanishing Newton step on a settled W: the multipliers of this step decide */
        if (!hard_release()) { done = 1; break; }
      }
    }
    /* the hard rows' solve did not settle within the iteration cap */
    if (nhard_act > 0 && !done && lane == 0) FB_FLAG_OR(g.flags, FB_FLAG_SOLVER);

    /* constraint forces */
    rows_apply(qacc, res);
    for (int r = lane; r < nrow; r += TEAM) {
      float rr = res[r] - aref[r];
      frc[r] = (rr < 0.f) ? -D[r]*rr : 0.f;
    }
    sync();
    /* a hard row's normal force lambda, a quarter on each of its four slots: J' frc adds Jn' lambda
     * and the contact force reads (lambda, 0, 0) */
    for (int h = lane; h < nhard_act; h += TEAM) {
      const int i = si[m.L.hcon + h];
      const float q = 0.25f*s[m.L.hlam + h];
      for (int k = 0; k < 4; k++) frc[2*nj + 4*i + k] = q;
    }
    if (nhard_act > 0) sync();
    rows_tapply(frc, fcon, 0);
    float *limf = s + m.L.limf;
    for (int j = lane; j < nj; j += TEAM) {
      /* jointlimitfrc = efc_force of the joint's first active limit row */
      limf[j] = D[2*j] > 0.f ? frc[2*j] : (D[2*j+1] > 0.f ? frc[2*j+1] : 0.f);
    }
    for (int i = lane; i < ncon; i += TEAM) {
      float mu = cand_mu(con_cand[i]);
      const float *f = frc + 2*nj + 4*i;
      g.d_con_force[3*i] = f[0] + f[1] + f[2] + f[3];
      g.d_con_force[3*i+1] = (f[0] - f[1])*mu;
      g.d_con_force[3*i+2] = (f[2] - f[3])*mu;
    }
    sync();
  }

  /* --------------------------------------- mj_forward for this state */
  FB_MEM void forward(int want_qacc) {
    const int nv = m.nv;
    float *fsm = s + m.L.fsm, *qacc = s + m.L.qacc, *fcon = s + m.L.fcon;
    kinematics();
    com_pos();
    com_vel_acc();
    body_forces_and_crb();
    mass_matrix_and_smooth();
    detect_constraints();
    for (int v = lane; v < nv; v += TEAM) fcon[v] = 0.f;
    int active = (nlim + ncon) > 0;
    if (active || want_qacc || !(m.any_damping || g.ep_damping)) {
      factor(0.f);
      for (int v = lane; v < nv; v += TEAM) qacc[v] = fsm[v];
      sync();
      solve_ld(qacc);
      if (active) {
        if (ncon > 0) make_contact_rows();
        solve_constraints(s + m.L.tmp1, s + m.L.tmp2);
      }
    }
    sync();
  }

  /* ------------------------------------------- A.10 Euler integrator */
  FB_MEM void euler() {
    const int nv = m.nv, nj = m.njnt;
    float *qpos = s + m.L.qpos, *qvel = s + m.L.qvel, *fsm = s + m.L.fsm, *fcon = s + m.L.fcon;
    float *x = s + m.L.grad;
    const float h = m.timestep;
    if (m.any_damping || g.ep_damping) {
      factor(h);
      for (int v = lane; v < nv; v += TEAM) x[v] = fsm[v] + fcon[v];
      sync();
      solve_ld(x);
    } else {
      const float *qacc = s + m.L.qacc;
      for (int v = lane; v < nv; v += TEAM) x[v] = qacc[v];
      sync();
    }
    for (int v = lane; v < nv; v += TEAM) qvel[v] += h*x[v];
    sync();
    int bad = 0;
    for (int j = lane; j < nj; j += TEAM) {
      int qa = MI(jnt_qposadr, j), da = MI(jnt_dofadr, j);
      if (MI(jnt_type, j) == FB_JNT_FREE) {
        for (int k = 0; k < 3; k++) qpos[qa + k] += h*qvel[da + k];
        float w[3] = {qvel[da + 3], qvel[da + 4], qvel[da + 5]};
        float angle = h*v_normalize3(w), sn, cs;
        fb_sincos(0.5f*angle, &sn, &cs);
        Quat qr = {cs, w[0]*sn, w[1]*sn, w[2]*sn};
        Quat q0 = {qpos[qa + 3], qpos[qa + 4], qpos[qa + 5], qpos[qa + 6]};
        Quat qn = q_normalize(q_mul(q_normalize(q0), qr));
        qpos[qa + 3] = qn.w; qpos[qa + 4] = qn.x; qpos[qa + 5] = qn.y; qpos[qa + 6] = qn.z;
        for (int k = 0; k < 7; k++) bad |= !(fabsf(qpos[qa + k]) < 1e30f);
      } else {
        qpos[qa] += h*qvel[da];
        bad |= !(fabsf(qpos[qa]) < 1e30f);
      }
    }
    if (bad) FB_FLAG_OR(g.flags, FB_FLAG_NONFINITE);
    sync();
  }

  /* ------------- physics2data + cycontacts2data + drag (fused log stage) */
  FB_MEM void body_velocity(int b, float *lin, float *ang) const {
    const int nb = m.nbody;
    const float *cvel = s + m.L.cvel, *xipos = s + m.L.xipos;
    ang[0] = cvel[b]; ang[1] = cvel[nb + b]; ang[2] = cvel[2*nb + b];
    float off[3] = {xipos[b] - comx, xipos[nb + b] - comy, xipos[2*nb + b] - comz}, cr[3];
    v_cross(ang, off, cr);
    lin[0] = cvel[3*nb + b] + cr[0]; lin[1] = cvel[4*nb + b] + cr[1]; lin[2] = cvel[5*nb + b] + cr[2];
  }

  FB_MEM void write_log() {
    const int nb = m.nbody, nj = m.njnt;
    const float *xpos = s + m.L.xpos, *xipos = s + m.L.xipos;
    const float *qpos = s + m.L.qpos, *qvel = s + m.L.qvel, *actf = s + m.L.actf;
    const float *limf = s + m.L.limf;
    float *xf = s + m.L.xfrc;
    /* links: physics.py:449-466 + :435-446 */
    for (int l = lane; l < m.n_links; l += TEAM) {
      int b = MI(link_body, l);
      Quat q = body_quat(b);
      float lin[3], ang[3];
      body_velocity(b, lin, ang);
      float *row = g.row_links + (long long)l*(20/FB_VEC_LINKS)*g.ev_links;
#define FB_L(c_) row[((c_)/FB_VEC_LINKS)*g.ev_links + ((c_) % FB_VEC_LINKS)]
      float im = m.inv_meters;
      FB_L(0) = xipos[b]*im; FB_L(1) = xipos[nb + b]*im; FB_L(2) = xipos[2*nb + b]*im;
      FB_L(3) = q.x; FB_L(4) = q.y; FB_L(5) = q.z; FB_L(6) = q.w;
      FB_L(7) = xpos[b]*im; FB_L(8) = xpos[nb + b]*im; FB_L(9) = xpos[2*nb + b]*im;
      FB_L(10) = q.x; FB_L(11) = q.y; FB_L(12) = q.z; FB_L(13) = q.w;
      FB_L(14) = lin[0]*m.inv_velocity; FB_L(15) = lin[1]*m.inv_velocity; FB_L(16) = lin[2]*m.inv_velocity;
      FB_L(17) = ang[0]*m.inv_angvel; FB_L(18) = ang[1]*m.inv_angvel; FB_L(19) = ang[2]*m.inv_angvel;
#undef FB_L
    }
    /* joints: physics.py:481-524 (the torque family is empty in the reference, D-4) */
    for (int j = lane; j < m.n_joints; j += TEAM) {
      float *row = g.row_joints + (long long)j*(m.joint_cols/FB_VEC_JOINTS)*g.ev_joints;
#define FB_J(c_) row[((c_)/FB_VEC_JOINTS)*g.ev_joints + ((c_) % FB_VEC_JOINTS)]
      for (int k = 0; k < m.joint_cols; k++) FB_J(k) = 0.f;
      FB_J(m.col_jpos) = qpos[MI(fj_qposadr, j)];
      FB_J(m.col_jvel) = qvel[MI(fj_dofadr, j)]*m.inv_angvel;
      float trq = 0.f;
      int ap = MI(fj_actpos, j), av = MI(fj_actvel, j), at = MI(fj_acttrq, j);
      if (ap >= 0) trq += actf[ap];
      if (av >= 0) trq += actf[av];
      if (at >= 0) trq += actf[at];
      FB_J(m.col_jtrq) = trq*m.inv_torques;
      int jid = MI(fj_jntid, j);
      FB_J(m.col_jlim) = jid >= 0 ? limf[jid]*m.inv_torques : 0.f;
#undef FB_J
    }
    /* contacts: sensors.pyx:140-190 */
    const int *con_cand = si + m.L.con_cand;
    for (int sx = lane; sx < m.n_contacts; sx += TEAM) {
      float acc[12], nsum = 0.f;
      for (int k = 0; k < 12; k++) acc[k] = 0.f;
      for (int i = 0; i < ncon; i++) {
        int c = con_cand[i];
        for (int key = 0; key < 4; key++) {
          if (MI(cand_sensor, 4*c + key) != sx) continue;
          float sg = (key & 1) ? 1.f : -1.f;
          float fn = g.d_con_force[3*i], f1 = g.d_con_force[3*i+1], f2 = g.d_con_force[3*i+2];
          const float *fr = g.d_con_frame + 9*i;
          float tot[3];
          for (int k = 0; k < 3; k++) {
            float re = sg*fn*fr[k], fri = sg*f1*fr[3+k] + sg*f2*fr[6+k];
            acc[k] += re; acc[3+k] += fri; tot[k] = re + fri; acc[6+k] += tot[k];
          }
          float nrm = sqrtf(tot[0]*tot[0] + tot[1]*tot[1] + tot[2]*tot[2]);
          for (int k = 0; k < 3; k++) acc[9+k] += nrm*g.d_con_pos[3*i + k];
          nsum += nrm;
        }
      }
      float *row = g.row_contacts + (long long)sx*(12/FB_VEC_CONTACTS)*g.ev_contacts;
#define FB_C(c_) row[((c_)/FB_VEC_CONTACTS)*g.ev_contacts + ((c_) % FB_VEC_CONTACTS)]
      float ip = nsum > 0.f ? 1.0f/nsum : 1.0f;
      for (int k = 0; k < 9; k++) FB_C(k) = acc[k]*m.inv_newtons;
      for (int k = 0; k < 3; k++) FB_C(9+k) = acc[9+k]*ip*m.inv_meters;
#undef FB_C
    }
    /* xfrc rows + xfrc_applied for the next step (drag.pyx:152-268, section 3.4) */
    for (int x = lane; x < m.n_xfrc; x += TEAM) {
      float *row = g.row_xfrc + (long long)x*(6/FB_VEC_XFRC)*g.ev_xfrc;
      for (int k = 0; k < 6; k++) row[(k/FB_VEC_XFRC)*g.ev_xfrc + (k % FB_VEC_XFRC)] = 0.f;
      int b = MI(xfrc_body, x);
      for (int k = 0; k < 6; k++) xf[k*nb + b] = 0.f;
    }
    sync();
    if (m.water_drag) {
      for (int i = lane; i < m.n_swim; i += TEAM) {
        int l = MI(swim_link, i), xi = MI(swim_xfrc, i), b = MI(link_body, l);
        float pz = xipos[2*nb + b]*m.inv_meters;
        if (pz > m.water_surface) continue;           /* drag.pyx:192-194 */
        float R[9], lin[3], ang[3], vl[3], wl[3], uw[3], buoy[3] = {0.f, 0.f, 0.f};
        q_mat(body_quat(b), R);
        body_velocity(b, lin, ang);
        m_rot_t(R, lin[0]*m.inv_velocity, lin[1]*m.inv_velocity, lin[2]*m.inv_velocity, vl);
        m_rot_t(R, ang[0]*m.inv_angvel, ang[1]*m.inv_angvel, ang[2]*m.inv_angvel, wl);
        float mass = MF(swim_mass, i);
        if (m.water_buoyancy && mass > 0.f && pz < m.water_surface) {
          float frac = fminf(fmaxf(m.water_surface - pz, 0.f)/MF(swim_height, i), 1.f);
          float lift = -1000.f*mass*(-9.81f)/MF(swim_density, i)*frac;
          m_rot_t(R, 0.f, 0.f, lift, buoy);
        }
        if (g.ep_wvel) m_rot_t(R, g.ep_wvel[0], g.ep_wvel[g.ep_pad], g.ep_wvel[2*g.ep_pad], uw);
        else m_rot_t(R, m.water_velocity[0], m.water_velocity[1], m.water_velocity[2], uw);
        float F[3], Tq[3];
        for (int k = 0; k < 3; k++) {
          float v = vl[k] - uw[k], w = wl[k];
          float sv = v < 0.f ? -v*v : v*v, sw = w < 0.f ? -w*w : w*w;
          const float cl = g.ep_coef ? g.ep_coef[(6*i + k)*g.ep_pad] : MF(swim_coef, 6*i + k);
          const float ca = g.ep_coef ? g.ep_coef[(6*i + 3 + k)*g.ep_pad] : MF(swim_coef, 6*i + 3 + k);
          F[k] = sv*m.water_viscosity*cl + buoy[k];
          Tq[k] = sw*ca;
        }
        float *row = g.row_xfrc + (long long)xi*(6/FB_VEC_XFRC)*g.ev_xfrc;
        for (int k = 0; k < 3; k++) {
          row[(k/FB_VEC_XFRC)*g.ev_xfrc + (k % FB_VEC_XFRC)] = F[k];
          row[((3+k)/FB_VEC_XFRC)*g.ev_xfrc + ((3+k) % FB_VEC_XFRC)] = Tq[k];
        }
        int bx = MI(xfrc_body, xi);
        float Rx[9], wf[3], wt[3];
        q_mat(body_quat(bx), Rx);
        m_rot(Rx, F[0], F[1], F[2], wf);
        m_rot(Rx, Tq[0], Tq[1], Tq[2], wt);
        for (int k = 0; k < 3; k++) { xf[k*nb + bx] = wf[k]*m.newtons; xf[(3+k)*nb + bx] = wt[k]*m.torques; }
      }
    }
    (void)nj;
    sync();
  }

  /* mjData-like derived quantities of the state the last forward() saw */
  FB_MEM void write_derived() {
    const int nb = m.nbody, nv = m.nv, nu = m.nu, nj = m.njnt;
    const float *xpos = s + m.L.xpos, *xipos = s + m.L.xipos;
    for (int b = lane; b < nb; b += TEAM) {
      Quat q = body_quat(b);
      float lin[3], ang[3];
      body_velocity(b, lin, ang);
      for (int k = 0; k < 3; k++) {
        g.d_xpos[3*b + k] = xpos[k*nb + b];
        g.d_xipos[3*b + k] = xipos[k*nb + b];
        g.d_linvel[3*b + k] = lin[k];
        g.d_angvel[3*b + k] = ang[k];
      }
      g.d_xquat[4*b] = q.w; g.d_xquat[4*b+1] = q.x; g.d_xquat[4*b+2] = q.y; g.d_xquat[4*b+3] = q.z;
    }
    for (int a = lane; a < nu; a += TEAM) g.d_actf[a] = (s + m.L.actf)[a];
    for (int j = lane; j < nj; j += TEAM) g.d_limf[j] = (s + m.L.limf)[j];
    for (int v = lane; v < nv; v += TEAM) g.d_qacc[v] = (s + m.L.qacc)[v];
  }

  /* on-device travelling-wave controller (replaces task.py:288-321 per-step Python) */
  FB_MEM void wave_control(float time) {
    float *ctrl = s + m.L.ctrl;
    for (int i = lane; i < m.n_wc; i += TEAM) {
      float ph = 6.283185307179586f*MF(wc_freq, i)*time - MF(wc_lag, i) + g.env_phase;
      ctrl[MI(wc_act, i)] = MF(wc_off, i) + MF(wc_amp, i)*sinf(ph);
    }
    sync();
  }

  /* ctrl of this step from the uploaded sequence (environment-minor) */
  FB_MEM void seq_control(const float *seq_env, long long env_pad) {
    float *ctrl = s + m.L.ctrl;
    for (int i = lane; i < m.nu; i += TEAM) ctrl[i] = seq_env[(long long)i*env_pad];
    sync();
  }

  FB_MEM void load_state() {
    float *qpos = s + m.L.qpos, *qvel = s + m.L.qvel, *ctrl = s + m.L.ctrl, *xf = s + m.L.xfrc;
    const int nb = m.nbody;
    for (int i = lane; i < m.nq; i += TEAM) qpos[i] = g.qpos[i];
    for (int i = lane; i < m.nv; i += TEAM) qvel[i] = g.qvel[i];
    for (int i = lane; i < m.nu; i += TEAM) ctrl[i] = g.ctrl[i];
    for (int i = lane; i < 6*nb; i += TEAM) { int b = i/6, k = i - 6*b; xf[k*nb + b] = g.xfrc_applied[i]; }
    sync();
  }

  FB_MEM void store_state(int ctrl_changed) {
    const float *qpos = s + m.L.qpos, *qvel = s + m.L.qvel, *ctrl = s + m.L.ctrl, *xf = s + m.L.xfrc;
    const int nb = m.nbody;
    for (int i = lane; i < m.nq; i += TEAM) g.qpos[i] = qpos[i];
    for (int i = lane; i < m.nv; i += TEAM) g.qvel[i] = qvel[i];
    if (m.n_wc > 0 || ctrl_changed) for (int i = lane; i < m.nu; i += TEAM) g.ctrl[i] = ctrl[i];
    for (int i = lane; i < 6*nb; i += TEAM) { int b = i/6, k = i - 6*b; g.xfrc_applied[i] = xf[k*nb + b]; }
  }
};

/* ===================================================================== */
/* launch parameters: device base pointers of the whole batch */
enum { FB_MODE_STEP = 0, FB_MODE_RESET = 1 };

struct FbParams {
  DevModel m;
  int n_envs, n_steps, ring, mode, want_derived;
  long long it0;                  /* batch iteration: physics steps taken since fb_reset */
  float *qpos, *qvel, *ctrl, *xfrc_applied, *qpos_spring, *env_phase;
  int *flags;
  long long *iteration;
  float *d_xpos, *d_xquat, *d_xipos, *d_linvel, *d_angvel, *d_actf, *d_limf, *d_qacc;
  int *d_ncon, *d_con_cand;
  float *d_con_dist, *d_con_pos, *d_con_frame, *d_con_force;
  float *J3, *efc, *prod3;
  /* device log, environment-minor (FbLogView): element (env, it, item, col) of a kind with N
   * items, C columns, vector width V at (((it*N + item)*(C/V) + col/V)*env_pad + env)*V + col%V */
  float *log_links, *log_joints, *log_contacts, *log_xfrc;
  long long env_pad;
  /* hand-over from the environment-per-thread kernel (fb_fast.h): environments that met
   * a limit or a contact, the step they stopped at, and how many there are.  The
   * counter is double-buffered by launch parity; use_pending = 0 -> every environment
   * from step 0. */
  int *pending, *pending_count, *steps_done;
  int use_pending, parity;
  /* control sequence (fb_set_ctrl_sequence): ctrl of step k of this launch is
   * ctrl_seq[((seq_pos + k)*nu + a)*env_pad + env]; NULL -> ctrl is held */
  const float *ctrl_seq;
  int seq_pos;
  /* rows of one sequence step: the nu ctrl values, then n_spring spring references (on-device CPG,
   * fb_set_cpg_springrefs: qpos_spring[spring_qadr[s]] of step k is row nu + s) */
  int seq_stride, n_spring;
  const int *spring_qadr;
  float *fast_scratch;            /* [n_scratch][fast_scratch_stride]: second half of the per-thread state */
  long long fast_scratch_stride;
  float *con_scratch;             /* per-thread constrained step (fb_fastc.h): [warp][X.n_con][lane] */
  /* Last iteration (row index before the ring modulus) at which a constraint-capable kernel wrote
   * this environment's log row, i.e. at which the contacts row / the joint_limit_force column may
   * be non-zero.  The unconstrained kernel zero-fills those columns only when the row it
   * overwrites was last written at or before that iteration (fb_fast.h: log_row_dirty); the
   * log starts zeroed (fb_create, fb_reset) and nothing else writes it. */
  long long *con_dirty;
  /* Groups of environments the SPLIT variant of the per-thread constrained kernel has stepped in
   * this launch (fb_fastc_split_kernel writes 0 / 1 per group; the single-warp kernel launched
   * behind it skips the groups marked 1).  NULL: the SPLIT variant was not launched. */
  int *con_split_done;
};

/* Per-environment parameter tables (fb_set_env_param), float32 environment-minor: value c of item i
 * of environment env at [(i*k + c)*env_pad + env] -- jnt_stiffness [njnt], dof_damping [nv], drag
 * coefficients [n_swim][6], water velocity [3], candidate friction [ncand].  NULL: the model's value
 * for every environment.
 * A launch argument of its own (not a member of FbParams), so that the parameter blocks of the
 * kernels that do not read it keep their layout: the team kernel tests the pointers at run time,
 * the per-thread kernels read them in their ENVP twins only (the unconstrained twins never read
 * `fric`: the member is last, so the members they read keep their offsets).
 * episode_start [n_envs] (fb_reset_envs): batch iteration of each environment's episode row 0; the
 * travelling-wave controller reads the episode's time (it0 + k - episode_start).  Bound only while
 * the wave controller is on and some episode began after iteration 0; NULL: it0 + k. */
struct FbEnvTables {
  const float *stiffness, *damping, *coef, *wvel;
  const float *fric;
  const long long *episode_start;
};

#define FB_NEVER_DIRTY (-(1LL << 60))

/* start of ring row `it` for one environment: floats_per_row = N*C of the kind */
FB_DEV float *fb_log_row(float *base, long long it, long long floats_per_row, long long env_pad, int vec,
                         size_t env) {
  return base + it*floats_per_row*env_pad + env*vec;
}

FB_DEV EnvPtrs fb_env_ptrs(const FbParams &P, const FbEnvTables &T, int env) {
  const DevModel &m = P.m;
  EnvPtrs g;
  size_t e = (size_t)env;
  g.qpos = P.qpos + e*m.nq; g.qvel = P.qvel + e*m.nv; g.ctrl = P.ctrl + e*(m.nu > 0 ? m.nu : 1);
  g.xfrc_applied = P.xfrc_applied + e*6*m.nbody; g.qpos_spring = P.qpos_spring + e*m.nq;
  g.env_phase = P.env_phase[env];
  g.flags = P.flags + env;
  g.d_xpos = P.d_xpos + e*3*m.nbody; g.d_xquat = P.d_xquat + e*4*m.nbody;
  g.d_xipos = P.d_xipos + e*3*m.nbody; g.d_linvel = P.d_linvel + e*3*m.nbody;
  g.d_angvel = P.d_angvel + e*3*m.nbody; g.d_actf = P.d_actf + e*(m.nu > 0 ? m.nu : 1);
  g.d_limf = P.d_limf + e*m.njnt; g.d_qacc = P.d_qacc + e*m.nv;
  int mc = m.maxcon > 0 ? m.maxcon : 1;
  g.d_ncon = P.d_ncon + env; g.d_con_cand = P.d_con_cand + e*mc;
  g.d_con_dist = P.d_con_dist + e*mc; g.d_con_pos = P.d_con_pos + e*3*mc;
  g.d_con_frame = P.d_con_frame + e*9*mc; g.d_con_force = P.d_con_force + e*3*mc;
  g.J3 = P.J3 + e*3*mc*m.nv; g.efc = P.efc + e*5*m.maxefc; g.prod3 = P.prod3 + e*6*mc;
  g.row_links = g.row_joints = g.row_contacts = g.row_xfrc = 0;
  g.ev_links = P.env_pad*FB_VEC_LINKS; g.ev_joints = P.env_pad*FB_VEC_JOINTS;
  g.ev_contacts = P.env_pad*FB_VEC_CONTACTS; g.ev_xfrc = P.env_pad*FB_VEC_XFRC;
  g.ep_stiffness = T.stiffness ? T.stiffness + e : 0;
  g.ep_damping = T.damping ? T.damping + e : 0;
  g.ep_coef = T.coef ? T.coef + e : 0;
  g.ep_wvel = T.wvel ? T.wvel + e : 0;
  g.ep_pad = P.env_pad;
  g.fric = T.fric ? T.fric + e : m.F + m.o.cand_friction;
  g.fric_stride = T.fric ? (int)P.env_pad : 1;
  return g;
}

/* Reset: forward at the loaded state, log row it0 % ring (0 after fb_reset; the episode's row 0 of
 * an environment fb_reset_envs restarts at it0).  Step k of a launch: control,
 * forward (derived quantities of the pre-step state), Euler, log row
 * (it0+k+1) % ring = {derived of the pre-step state, qpos/qvel of the new
 * state} (SURVEY.md Appendix D-1), then the drag wrench for the next step. */
template <int TEAM>
FB_DEV void fb_run_env(const FbParams &P, const FbEnvTables &T, int env, int k0, float *s, int *si, int lane, int base,
                       unsigned mask) {
  const DevModel &m = P.m;
  FbStep<TEAM> st(m, s, si, fb_env_ptrs(P, T, env), lane, base, mask);
  st.init_world();
  st.load_state();
  const size_t e = (size_t)env;
  const int n = P.mode == FB_MODE_RESET ? 1 : P.n_steps;
  for (int k = k0; k < n; k++) {
    long long row;
    if (P.mode == FB_MODE_RESET) {
      st.forward(1);
      row = P.it0 % P.ring;
    } else {
      if (P.ctrl_seq) {
        const float *seqk = P.ctrl_seq + ((size_t)(P.seq_pos + k)*P.seq_stride)*P.env_pad + e;
        /* model.qpos_spring of this step (task.py:338-346), before forward() reads it */
        for (int i = lane; i < P.n_spring; i += TEAM) st.g.qpos_spring[P.spring_qadr[i]] = seqk[(long long)(m.nu + i)*P.env_pad];
        st.seq_control(seqk, P.env_pad);
      }
      if (m.n_wc > 0) st.wave_control((float)(P.it0 + k - (T.episode_start ? T.episode_start[e] : 0))*m.timestep);
      int wd = P.want_derived && k == n - 1;
      st.forward(wd);
      if (wd) st.write_derived();
      st.euler();
      row = (P.it0 + k + 1) % P.ring;
    }
    st.g.row_links = fb_log_row(P.log_links, row, m.n_links*20, P.env_pad, FB_VEC_LINKS, e);
    st.g.row_joints = fb_log_row(P.log_joints, row, m.n_joints*m.joint_cols, P.env_pad, FB_VEC_JOINTS, e);
    st.g.row_contacts = fb_log_row(P.log_contacts, row, m.n_contacts*12, P.env_pad, FB_VEC_CONTACTS, e);
    st.g.row_xfrc = fb_log_row(P.log_xfrc, row, m.n_xfrc*6, P.env_pad, FB_VEC_XFRC, e);
    st.write_log();
    if (P.mode == FB_MODE_RESET) st.write_derived();
  }
  st.store_state(P.ctrl_seq != 0 && P.mode != FB_MODE_RESET);
  if (lane == 0) {
    P.iteration[env] = P.mode == FB_MODE_RESET ? P.it0 : P.it0 + P.n_steps;
    if (k0 < n) P.con_dirty[env] = P.mode == FB_MODE_RESET ? P.it0 : P.it0 + P.n_steps;   /* full rows, constraint columns included */
  }
}

#endif /* FB_DEVICE_H_ */
