/*
 * fb_engine.cu -- C ABI (include/farms_b200.h) of the batched FARMS stepping
 * engine and its CUDA kernels for sm_100a.
 *
 * One CUDA thread TEAM (8/16/32 lanes of a warp) steps one environment; the
 * environment's working set is staged in shared memory for the n_steps of a
 * launch, so HBM only sees the initial/final state and the farms log rows.
 *
 * Built as the product with nvcc (-gencode arch=compute_100a,code=sm_100a).
 * The same file compiles with g++ -DFB_HOST_EMU into tests/emu/libfb_emu.so, a
 * unit-test harness that runs the device code serially on the host (TEAM = 1)
 * so the arithmetic can be checked on the GPU-less development box.  The
 * product never loads that library.
 */
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <new>
#include <string>
#include <type_traits>
#include <vector>
#ifdef FB_HOST_EMU
#include <thread>
#endif

#include "fb_fastc.h"
#include "fb_cpg.h"
#include "fb_drag.h"

#ifndef FB_HOST_EMU
#include <cuda_runtime.h>
#endif

static thread_local std::string g_error;
static int fail(const std::string &msg) { g_error = msg; return -1; }

/* ------------------------------------------------------- memory backend */
#ifdef FB_HOST_EMU
typedef int fbStream;
static int dev_alloc(void **p, size_t bytes) { *p = calloc(bytes ? bytes : 1, 1); return *p ? 0 : -1; }
static void dev_free(void *p) { free(p); }
static int dev_zero(void *p, size_t bytes, fbStream) { memset(p, 0, bytes); return 0; }
static int h2d(void *d, const void *h, size_t bytes, fbStream) { memcpy(d, h, bytes); return 0; }
static int d2h(void *h, const void *d, size_t bytes, fbStream) { memcpy(h, d, bytes); return 0; }
static int dev_sync(fbStream) { return 0; }
static const char *dev_error() { return "emulation backend error"; }
#else
typedef cudaStream_t fbStream;
static int dev_alloc(void **p, size_t bytes) {
  if (cudaMalloc(p, bytes ? bytes : 1) != cudaSuccess) return -1;
  /* the memset runs on the legacy stream, which the handle's non-blocking
   * stream does not order against: wait for it before anyone uploads */
  if (cudaMemset(*p, 0, bytes ? bytes : 1) != cudaSuccess) return -1;
  return cudaDeviceSynchronize() == cudaSuccess ? 0 : -1;
}
static void dev_free(void *p) { cudaFree(p); }
static int dev_zero(void *p, size_t bytes, fbStream st) { return cudaMemsetAsync(p, 0, bytes, st) == cudaSuccess ? 0 : -1; }
static int h2d(void *d, const void *h, size_t bytes, fbStream st) { return cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, st) == cudaSuccess ? 0 : -1; }
static int d2h(void *h, const void *d, size_t bytes, fbStream st) { return cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, st) == cudaSuccess ? 0 : -1; }
static int dev_sync(fbStream st) { return cudaStreamSynchronize(st) == cudaSuccess ? 0 : -1; }
static const char *dev_error() { return cudaGetErrorString(cudaGetLastError()); }
#endif

/* fb_reset_envs: what a restart writes besides the reset's forward pass (the team kernel's) */
struct FbResetArgs {
  const uint8_t *mask;             /* [n_envs] non-zero: restart */
  const float *qpos0, *qvel0;      /* given rows ([row][nq] / [row][nv]) or NULL: the keyframe */
  const int *row_of;               /* [n_envs] row of qpos0 / qvel0 of a restarted environment; NULL: env */
  const float *key_qpos, *key_qvel;
  float *qpos, *qvel, *ctrl, *xfrc_applied;
  int *flags;
  long long *episode_start;
  float *theta, *r, *rd;           /* on-device CPG state [n_osc][env_pad] (n_osc = 0: no CPG) */
  const float *theta0, *r0;        /* ... as fb_set_cpg_state last set it */
  int n_envs, nq, nv, nu, nbody, n_osc;
  long long env_pad, it;
};

/* one environment: its state rows as fb_reset writes them, its CPG rows, its episode start */
FB_DEV void fb_reset_env(const FbResetArgs &A, int env) {
  if (!A.mask[env]) return;
  const size_t e = (size_t)env, row = A.row_of ? (size_t)A.row_of[env] : e;
  for (int i = 0; i < A.nq; i++) A.qpos[e*A.nq + i] = A.qpos0 ? A.qpos0[row*A.nq + i] : A.key_qpos[i];
  for (int i = 0; i < A.nv; i++) A.qvel[e*A.nv + i] = A.qvel0 ? A.qvel0[row*A.nv + i] : A.key_qvel[i];
  const int nu = A.nu > 0 ? A.nu : 1;
  for (int i = 0; i < nu; i++) A.ctrl[e*nu + i] = 0.f;
  for (int i = 0; i < 6*A.nbody; i++) A.xfrc_applied[e*6*A.nbody + i] = 0.f;
  A.flags[env] = 0;
  for (int o = 0; o < A.n_osc; o++) {
    const size_t k = (size_t)o*A.env_pad + e;
    A.theta[k] = A.theta0[k]; A.r[k] = A.r0[k]; A.rd[k] = 0.f;
  }
  A.episode_start[env] = A.it;
}

/* --------------------------------------------------------------- kernels */
/* behind the body blocks of a SPLIT block: root position [3][32] + hand-over flags [32] ... */
#define FB_SPLIT_EXTRA_BYTES 512
/* ... and of a constrained SPLIT block, floats per lane: root position [3], hand-over flag, reduction buffers */
#define FB_CSPLIT_EXTRA (4 + 2*FB_SPLIT_MAXW*FB_RED_MAX)
#ifndef FB_HOST_EMU
/* only: FB_MODE_RESET of fb_reset_envs, the environments to restart ([n_envs], non-zero); NULL: all */
template <int TEAM>
__global__ void __launch_bounds__(128)
fb_step_kernel(const __grid_constant__ FbParams P, const __grid_constant__ FbEnvTables T, const uint8_t *only) {
  extern __shared__ __align__(16) float fb_smem[];
  const DevModel &m = P.m;
  const int tid = threadIdx.x, team = tid/TEAM, lane = tid % TEAM;
  int env = blockIdx.x*(blockDim.x/TEAM) + team, k0 = 0;
  if (P.use_pending) {
    /* only the environments the per-thread kernel handed over, from the step they stopped at */
    if (env >= P.pending_count[P.parity]) return;
    env = P.pending[env];
    k0 = P.steps_done[env];
  } else if (env >= P.n_envs || (only && !only[env])) {
    return;
  }
  const int base = (tid & 31)/TEAM*TEAM;
  const unsigned mask = TEAM == 32 ? 0xffffffffu : (((1u << (TEAM & 31)) - 1u) << base);
  float *s = fb_smem + (size_t)team*(m.L.n_float + m.L.n_int);
  int *si = reinterpret_cast<int *>(s + m.L.n_float);
  fb_run_env<TEAM>(P, T, env, k0, s, si, lane, base, mask);
}

/* environment-per-thread kernel (fb_fast.h): no barriers, no shuffles; BLK threads =
 * BLK environments whose working sets interleave in shared memory */
struct FbFastParams {
  FbParams P;
  FastRec rec[FB_FAST_MAXBODY];   /* per-body records, read from the constant bank */
};

/* Every per-thread kernel takes ENVP as its last template argument.  ENVP = 1 reads the
 * per-environment parameter tables of fb_set_env_param and runs the episode clock of fb_reset_envs;
 * its parameters are the ENVP = 0 struct with the tables appended (Fb*EnvParams), so the ENVP = 0
 * layouts stay as they are.  fb_plan picks ENVP = 1 while a table the kernel reads is set or the
 * episode clock is bound.  Each body is written out inside its __global__ function rather than
 * called as an inlined function, which ptxas was found to schedule differently. */
template <int ENVP, class Q> FB_DEV const FbEnvTables *fb_env_tables(const Q &q) {
  if constexpr (ENVP != 0) return &q.T; else return nullptr;
}
struct FbFastEnvParams : FbFastParams { FbEnvTables T; };

/* BLK environments per warp (32, or 16 in a half-filled warp).  MULTI: blocks of 2..8 warps
 * (blockDim.x/32) kept in step by a barrier per physics step (FbFast::run_t). */
template <int BLK, int SLIM, int MULTI, int LEAN, int ENVP>
__global__ void __launch_bounds__(MULTI ? 256 : 32)
fb_fast_kernel(const __grid_constant__ std::conditional_t<ENVP != 0, FbFastEnvParams, FbFastParams> Q) {
  extern __shared__ __align__(16) float fb_smem[];
  const FbParams &P = Q.P;
  const int warp = MULTI ? threadIdx.x >> 5 : 0, lane = MULTI ? threadIdx.x & 31 : threadIdx.x;
  const int wid = MULTI ? blockIdx.x*(blockDim.x >> 5) + warp : blockIdx.x;   /* warp index of the launch */
  const int env = wid*BLK + lane;
  if (blockIdx.x == 0 && threadIdx.x == 0) P.pending_count[P.parity ^ 1] = 0;   /* for the next launch */
  const int valid = env < P.n_envs;
  if (!MULTI && !valid) return;
  const int n_float = SLIM ? P.m.X.n_float_slim : P.m.X.n_float;
  const size_t warp_floats = (size_t)n_float*BLK;
  /* L2-resident scratch [warp][field][lane]: compile-time strides, coalesced */
  FbFast<BLK, SLIM, LEAN, 0, ENVP> st(P, Q.rec, fb_smem + warp*warp_floats + lane,
                             P.fast_scratch + (size_t)wid*(SLIM ? P.m.X.n_scratch_slim : P.m.X.n_scratch)*BLK + lane,
                             valid ? env : 0, fb_env_tables<ENVP>(Q));
  /* full warps move their state through a shared-memory tile (coalesced); a partial last
   * warp, or a model whose state rows do not fit the tile, uses per-thread accesses (the SLIM
   * layout's smaller blocks take the rows in two phases) */
  const int coop = BLK == 32 && (wid + 1)*BLK <= P.n_envs ? (SLIM ? 2*P.m.X.coop_io2 : P.m.X.coop_io) : 0;
  const int done = st.template run_t<MULTI>(coop, lane, valid);
  if (valid && done < P.n_steps) {
    P.steps_done[env] = done;
    P.pending[atomicAdd(P.pending_count + P.parity, 1)] = env;
  }
}

/* SPLIT variant (small batches): one block = 32 environments stepped by split.nwarps warps */
struct FbFastSplitParams {
  FbParams P;
  FastRec rec[FB_FAST_MAXBODY];
  FastSplit split;
};

/* registers capped for 3 blocks of 128 threads per SM (168): with the 96-thread blocks of a
 * three-way split four blocks are then resident (shared memory allows four), i.e. 592 blocks =
 * 18,944 environments in one wave.  Measured r2t (SALAMANDER, 16 steps per launch): 12,288 envs
 * 0.82 ms, 16,384 envs 0.83 ms; uncapped (197 registers, 2 blocks per SM) 1.42 ms beyond 9,472
 * envs; capped for 4 blocks of 128 (128 registers, spills) 1.07 .. 1.13 ms. */
#ifndef FB_SPLIT_MINBLOCKS
#define FB_SPLIT_MINBLOCKS 3
#endif
struct FbFastSplitEnvParams : FbFastSplitParams { FbEnvTables T; };
template <int LEAN, int ENVP>
__global__ void __launch_bounds__(32*FB_SPLIT_MAXW, FB_SPLIT_MINBLOCKS)
fb_fast_split_kernel(const __grid_constant__ std::conditional_t<ENVP != 0, FbFastSplitEnvParams, FbFastSplitParams> Q) {
  extern __shared__ __align__(16) float fb_smem[];
  const FbParams &P = Q.P;
  const int role = threadIdx.x >> 5, lane = threadIdx.x & 31, wid = blockIdx.x;
  const int env = wid*32 + lane;
  if (blockIdx.x == 0 && threadIdx.x == 0) P.pending_count[P.parity ^ 1] = 0;   /* for the next launch */
  const int valid = env < P.n_envs;
  const int n_float = P.m.X.n_float;
  FbFast<32, 0, LEAN, 1, ENVP> st(P, Q.rec, fb_smem + lane, P.fast_scratch + (size_t)wid*P.m.X.n_scratch*32 + lane,
                            valid ? env : 0, fb_env_tables<ENVP>(Q));
  float *extra = fb_smem + (size_t)n_float*32;
  st.split_setup(Q.split, role, extra + lane, reinterpret_cast<int *>(extra + 3*32) + lane);
  const int coop = (wid + 1)*32 <= P.n_envs ? P.m.X.coop_io : 0;
  const int done = st.run_split(coop, lane, valid);
  if (role == 0 && valid && done < P.n_steps) {
    P.steps_done[env] = done;
    P.pending[atomicAdd(P.pending_count + P.parity, 1)] = env;
  }
}

struct FbFastConParams {
  FbParams P;
  FastRec rec[FB_FAST_MAXBODY];
  CandRec cand[FB_FAST_MAXCAND];  /* collision candidates in body order, constant bank */
};
static_assert(sizeof(FbFastConParams) <= 32764, "kernel parameters of fb_fastc_kernel exceed 32 KB");

struct FbFastConEnvParams : FbFastConParams { FbEnvTables T; };
static_assert(sizeof(FbFastConEnvParams) <= 32764, "kernel parameters of fb_fastc_kernel<..., 1> exceed 32 KB");
template <int BLK, int LEAN, int ENVP>
__global__ void __launch_bounds__(BLK)
fb_fastc_kernel(const __grid_constant__ std::conditional_t<ENVP != 0, FbFastConEnvParams, FbFastConParams> Q) {
  extern __shared__ __align__(16) float fb_smem[];
  const FbParams &P = Q.P;
  const int i = blockIdx.x*BLK + threadIdx.x;
  const int count = P.use_pending ? P.pending_count[P.parity] : P.n_envs;
  if (i >= count) return;
  if (P.con_split_done && P.con_split_done[blockIdx.x]) return;      /* stepped by the SPLIT variant */
  const int identity = !P.use_pending || count == P.n_envs;
  const int env = identity ? i : P.pending[i];
  const int k0 = P.use_pending ? P.steps_done[env] : 0;
  const size_t t0 = (size_t)blockIdx.x*BLK;
  FbFastCon<BLK, LEAN, 0, ENVP> st(P, Q.rec, Q.cand, fb_smem + threadIdx.x, P.fast_scratch + t0*P.m.X.n_scratch + threadIdx.x,
                    P.con_scratch + t0*P.m.X.n_con + threadIdx.x, env, fb_env_tables<ENVP>(Q));
  const int coop = BLK == 32 && identity && P.m.X.coop_io && (blockIdx.x + 1)*BLK <= count;
  st.run_con(k0, coop, threadIdx.x);
}

/* SPLIT variant of the constrained kernel: one block = the BLK environments of one group (the
 * lanes of a warp; the upper half-warp leaves at once when BLK = 16) stepped by split.nwarps
 * warps, each its own bodies of the tree.  It takes the groups in which EVERY environment was
 * handed over before its first step (ground-contact batches: all of them, every launch) and marks
 * them in con_split_done; everything else is left to fb_fastc_kernel, launched behind it. */
struct FbFastConSplitParams {
  FbParams P;
  FastRec rec[FB_FAST_MAXBODY];
  CandRec cand[FB_FAST_MAXCAND];
  FastSplit split;
};
static_assert(sizeof(FbFastConSplitParams) <= 32764, "kernel parameters of fb_fastc_split_kernel exceed 32 KB");
#ifndef FB_CSPLIT_MINBLOCKS
#define FB_CSPLIT_MINBLOCKS 2
#endif
struct FbFastConSplitEnvParams : FbFastConSplitParams { FbEnvTables T; };
static_assert(sizeof(FbFastConSplitEnvParams) <= 32764, "kernel parameters of fb_fastc_split_kernel<..., 1> exceed 32 KB");
template <int BLK, int LEAN, int ENVP>
__global__ void __launch_bounds__(32*FB_SPLIT_MAXW, FB_CSPLIT_MINBLOCKS)
fb_fastc_split_kernel(const __grid_constant__ std::conditional_t<ENVP != 0, FbFastConSplitEnvParams, FbFastConSplitParams> Q) {
  extern __shared__ __align__(16) float fb_smem[];
  const FbParams &P = Q.P;
  const int role = threadIdx.x >> 5, lane = threadIdx.x & 31, grp = blockIdx.x;
  const int env = grp*BLK + lane;
  if (lane >= BLK || env >= P.n_envs) return;
  /* block-uniform: every warp sees the same lanes */
  const int all0 = P.pending_count[P.parity] == P.n_envs && __ballot_sync(__activemask(), P.steps_done[env] != 0) == 0u;
  if (threadIdx.x == 0) P.con_split_done[grp] = all0;
  if (!all0) return;
  const size_t t0 = (size_t)grp*BLK;
  FbFastCon<BLK, LEAN, 1, ENVP> st(P, Q.rec, Q.cand, fb_smem + lane, P.fast_scratch + t0*P.m.X.n_scratch + lane,
                             P.con_scratch + t0*P.m.X.n_con + lane, env, fb_env_tables<ENVP>(Q));
  float *extra = fb_smem + (size_t)P.m.X.n_float*BLK;
  st.split_setup(Q.split, role, extra + lane, reinterpret_cast<int *>(extra + 3*BLK) + lane);
  st.con_split_setup(Q.split, extra + 4*BLK + lane);
  const int coop = BLK == 32 && P.m.X.coop_io && (grp + 1)*BLK <= P.n_envs;
  st.run_con_split(coop, lane);
}

/* Stand-alone drag operator (fb_drag_forces, fb_drag.h): one thread = one link row */
__global__ void __launch_bounds__(128) fb_drag_forces_kernel(const FbDragArgs A) {
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if (i < A.n) fb_drag_row(A, i);
}

/* ring row `row` of every environment -> dense [n_envs][row_floats] (the reference's row
 * layout); threads run over (vector, env) with env fastest: coalesced reads */
__global__ void fb_gather_rows_kernel(const float *__restrict__ log, long long row, int row_floats,
                                      int vec, long long env_pad, int n_envs, float *__restrict__ out) {
  long long i = (long long)blockIdx.x*blockDim.x + threadIdx.x;
  const int nvec = row_floats/vec;
  if (i >= (long long)nvec*n_envs) return;
  const long long g = i/n_envs, env = i - g*n_envs;
  const float *src = log + ((row*nvec + g)*env_pad + env)*vec;
  float *dst = out + env*row_floats + g*vec;
  for (int k = 0; k < vec; k++) dst[k] = src[k];
}

/* Plain copy by the SMs, 16 bytes per access when both ends allow it.  fb_step_host uses it to
 * read ctrl straight out of PINNED host memory (mapped under unified addressing): a
 * cudaMemcpyAsync upload shares the copy-engine queue with the row download of the previous
 * launch and was measured to wait for it (up + down 7.1 ms per launch against 3.7 either way). */
__global__ void __launch_bounds__(256) fb_copy_kernel(const float *__restrict__ src, float *__restrict__ dst,
                                                      long long n, int vec4) {
  const long long stride = (long long)gridDim.x*blockDim.x, t = (long long)blockIdx.x*blockDim.x + threadIdx.x;
  if (vec4) {
    const float4 *s4 = reinterpret_cast<const float4 *>(src);
    float4 *d4 = reinterpret_cast<float4 *>(dst);
    const long long n4 = n >> 2;
    long long i = t;
    for (; i + 3*stride < n4; i += 4*stride) {          /* four loads in flight per thread */
      const float4 a = s4[i], b = s4[i + stride], c = s4[i + 2*stride], d = s4[i + 3*stride];
      d4[i] = a; d4[i + stride] = b; d4[i + 2*stride] = c; d4[i + 3*stride] = d;
    }
    for (; i < n4; i += stride) d4[i] = s4[i];
    for (long long k = (n4 << 2) + t; k < n; k += stride) dst[k] = src[k];
  } else {
    for (long long i = t; i < n; i += stride) dst[i] = src[i];
  }
}

/* The same for 4-float vectors (the links log) through a shared-memory tile of 32 environments x
 * 32 vectors: reads run along the environments (512 contiguous bytes per warp, as the log is
 * laid out), writes along the row (512 contiguous bytes of one environment's dense row). */
__global__ void __launch_bounds__(256) fb_gather_rows4_kernel(const float4 *__restrict__ log4, long long row, int nvec,
                                                              long long env_pad, int n_envs, float4 *__restrict__ out4) {
  __shared__ float4 tile[32][33];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int env0 = blockIdx.x*32, g0 = blockIdx.y*32;
  for (int g = w; g < 32; g += 8)
    if (g0 + g < nvec && env0 + lane < n_envs) tile[g][lane] = log4[(row*nvec + g0 + g)*env_pad + env0 + lane];
  __syncthreads();
  for (int e = w; e < 32; e += 8)
    if (env0 + e < n_envs && g0 + lane < nvec) out4[(long long)(env0 + e)*nvec + g0 + lane] = tile[lane][e];
}

/* selected columns of ring row `row` of every environment -> dense [n_envs][n_items][n_sel] */
/* n_sel_items > 0: only the listed items (fb_set_host_link_items), else all n_items */
struct FbColSel { int n; int col[32]; int n_sel_items; int item[64]; };
__global__ void fb_gather_cols_kernel(const float *__restrict__ log, long long row, int n_items, int n_cols,
                                      int vec, long long env_pad, int n_envs, FbColSel sel,
                                      float *__restrict__ out) {
  long long i = (long long)blockIdx.x*blockDim.x + threadIdx.x;
  const int out_items = sel.n_sel_items > 0 ? sel.n_sel_items : n_items;
  const long long per_env = (long long)out_items*sel.n;
  if (i >= per_env*n_envs) return;
  const long long k = i/n_envs, env = i - k*n_envs;            /* env fastest: coalesced reads */
  const int oi = (int)(k/sel.n), c = sel.col[k - (long long)oi*sel.n];
  const int item = sel.n_sel_items > 0 ? sel.item[oi] : oi;
  const long long f = (long long)item*n_cols + c, nvec = (long long)n_items*n_cols/vec;
  out[env*per_env + k] = log[((row*nvec + f/vec)*env_pad + env)*vec + f % vec];
}

/* uploaded ctrl columns [n_envs][n_sel] -> ctrl[n_envs][nu] at the selected actuators */
__global__ void fb_scatter_ctrl_kernel(const float *__restrict__ in, int n_envs, int nu, FbColSel sel,
                                       float *__restrict__ ctrl) {
  long long i = (long long)blockIdx.x*blockDim.x + threadIdx.x;
  if (i >= (long long)n_envs*sel.n) return;
  const long long env = i/sel.n;
  ctrl[env*nu + sel.col[i - env*sel.n]] = in[i];
}

/* control sequence [K][n_envs][nu] (host order) -> [K][nu][env_pad] (environment-minor) */
__global__ void fb_transpose_ctrl_kernel(const float *__restrict__ in, int K, int n_envs, int nu,
                                         long long env_pad, float *__restrict__ out) {
  long long i = (long long)blockIdx.x*blockDim.x + threadIdx.x;
  if (i >= (long long)K*nu*n_envs) return;
  const long long env = i % n_envs, ka = i/n_envs;          /* ka = k*nu + a */
  const long long k = ka/nu, a = ka - k*nu;
  out[ka*env_pad + env] = in[(k*n_envs + env)*nu + a];
}

/* on-device CPG (fb_cpg.h): the control vectors of the launch's n_steps, one thread per environment */
__global__ void __launch_bounds__(128) fb_cpg_kernel(CpgDev c, int n_envs, long long env_pad, int n_steps, int nu,
                                                      float dt, const float *__restrict__ ctrl, float *__restrict__ seq) {
  const int env = blockIdx.x*blockDim.x + threadIdx.x;
  if (env < n_envs) fb_cpg_env(c, env, env_pad, n_steps, nu, dt, ctrl, seq);
}

/* fb_reset_envs_where: one thread per environment */
__global__ void __launch_bounds__(128) fb_reset_envs_kernel(const FbResetArgs A) {
  const int env = blockIdx.x*blockDim.x + threadIdx.x;
  if (env < A.n_envs) fb_reset_env(A, env);
}

/* fb_reset_envs: the host list envs[n] -> mask (zeroed before) and the row of each listed environment */
__global__ void fb_reset_list_kernel(const int *__restrict__ envs, int n, uint8_t *mask, int *row_of) {
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if (i < n) { mask[envs[i]] = 1; row_of[envs[i]] = i; }
}

/* the whole ring of one environment -> dense [ring][row_floats] */
__global__ void fb_gather_env_kernel(const float *__restrict__ log, int ring, int row_floats, int vec,
                                     long long env_pad, int env, float *__restrict__ out) {
  long long i = (long long)blockIdx.x*blockDim.x + threadIdx.x;
  if (i >= (long long)ring*row_floats) return;
  const long long lin = i/vec;       /* (it*nvec + g) */
  out[i] = log[(lin*env_pad + env)*vec + (i - lin*vec)];
}
#endif

/* ------------------------------------------------------ per-thread kernel variants */
enum { FB_FAST, FB_FAST_SPLIT, FB_FASTC, FB_FASTC_SPLIT };      /* FbKernelSel::kind */

/* One per-thread kernel launch: the instantiation and its shape.  FB_FAST covers the regular
 * layout (BLK = 32 or 16), SLIM (BLK = 32) and SLIM in blocks of threads/32 warps (MULTI);
 * BLK of the constrained kernels is the environments per group. */
struct FbKernelSel {
  int kind, blk, slim, multi, lean, envp;
  int grid, threads;
  size_t bytes;
};

template <int KIND, int BLK, int SLIM, int MULTI, int LEAN, int ENVP> struct FbVariant {
  static constexpr int kind = KIND, blk = BLK, slim = SLIM, multi = MULTI, lean = LEAN, envp = ENVP;
};
template <int KIND, int BLK, int SLIM, int MULTI, class F> static void fb_dispatch_le(const FbKernelSel &k, F &f) {
  if (k.lean) {
    if (k.envp) f(FbVariant<KIND, BLK, SLIM, MULTI, 1, 1>()); else f(FbVariant<KIND, BLK, SLIM, MULTI, 1, 0>());
  } else {
    if (k.envp) f(FbVariant<KIND, BLK, SLIM, MULTI, 0, 1>()); else f(FbVariant<KIND, BLK, SLIM, MULTI, 0, 0>());
  }
}
/* The per-thread kernels built, each with LEAN x ENVP: calls f(FbVariant<...>()) for the one `k`
 * selects.  Every launch, attribute and occupancy query of a per-thread kernel, and the emulation
 * (which runs each variant with BLK = 1), goes through here. */
template <class F> static void fb_dispatch(const FbKernelSel &k, F &&f) {
  switch (k.kind) {
    case FB_FAST:
      if (k.blk == 16) fb_dispatch_le<FB_FAST, 16, 0, 0>(k, f);
      else if (!k.slim) fb_dispatch_le<FB_FAST, 32, 0, 0>(k, f);
      else if (!k.multi) fb_dispatch_le<FB_FAST, 32, 1, 0>(k, f);
      else fb_dispatch_le<FB_FAST, 32, 1, 1>(k, f);
      break;
    case FB_FAST_SPLIT: fb_dispatch_le<FB_FAST_SPLIT, 32, 0, 0>(k, f); break;
    case FB_FASTC:
      if (k.blk == 16) fb_dispatch_le<FB_FASTC, 16, 0, 0>(k, f); else fb_dispatch_le<FB_FASTC, 32, 0, 0>(k, f);
      break;
    default:
      if (k.blk == 16) fb_dispatch_le<FB_FASTC_SPLIT, 16, 0, 0>(k, f); else fb_dispatch_le<FB_FASTC_SPLIT, 32, 0, 0>(k, f);
      break;
  }
}

#ifndef FB_HOST_EMU
template <class V> static auto fb_kernel_of(V) {
  if constexpr (V::kind == FB_FAST) return fb_fast_kernel<V::blk, V::slim, V::multi, V::lean, V::envp>;
  else if constexpr (V::kind == FB_FAST_SPLIT) return fb_fast_split_kernel<V::lean, V::envp>;
  else if constexpr (V::kind == FB_FASTC) return fb_fastc_kernel<V::blk, V::lean, V::envp>;
  else return fb_fastc_split_kernel<V::blk, V::lean, V::envp>;
}

/* The shared-memory attributes of the four LEAN x ENVP instantiations of `k` for k.bytes and, with
 * per_sm, the fewest blocks of k.threads of them an SM holds */
static cudaError_t fb_kernel_attributes(FbKernelSel k, int *per_sm = nullptr) {
  cudaError_t ce = cudaSuccess;
  if (per_sm) *per_sm = 1 << 30;
  for (int v = 0; v < 4 && ce == cudaSuccess; v++) {
    k.lean = v & 1; k.envp = v >> 1;
    fb_dispatch(k, [&](auto var) {
      const void *f = (const void *)fb_kernel_of(var);
      ce = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.bytes);
      if (ce == cudaSuccess) ce = cudaFuncSetAttribute(f, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
      int nb = 0;
      if (ce == cudaSuccess && per_sm) ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, f, k.threads, k.bytes);
      if (per_sm && nb < *per_sm) *per_sm = nb;
    });
  }
  return ce;
}

/* the team kernel of `team` lanes per environment */
typedef void (*FbTeamKernel)(FbParams, FbEnvTables, const uint8_t *);
static FbTeamKernel fb_team_kernel(int team) {
  switch (team) {
    case 8: return fb_step_kernel<8>;
    case 16: return fb_step_kernel<16>;
    default: return fb_step_kernel<32>;
  }
}
#endif

/* ---------------------------------------------------------------- handle */
enum { FB_N_ENV_PARAM = FB_ENV_ACT_BIAS + 1 };     /* fields of fb_set_env_param */

struct FbHandle {
  FbHostModel hm;
  FbParams P;
  int device, team, envs_per_block, threads;
  size_t smem_bytes;
  int fast_enabled, fast_block;     /* environment-per-thread kernel: on/off, threads per block */
  int con_thread;                   /* 1: hand-overs go to the per-thread constrained kernel, 0: to the team kernel */
  int fast_slim;                    /* 1: SLIM layout of the unconstrained kernel (8 warps per SM; large batches) */
  int fast_wpb;                     /* warps per block of the unconstrained kernel (> 1: barrier per step) */
  int fast_lean;                    /* 1: use the LEAN variants when the model allows (FARMS_B200_FAST_LEAN=0 switches them off) */
  int fast_split;                   /* 1: small batches run the SPLIT variant (several warps per 32 environments) */
  long long split_capacity;         /* blocks of the SPLIT variant the device holds at once (0: not applicable) */
  int con_split;                    /* 1: ground-contact batches run the SPLIT variant of the constrained kernel */
  long long con_split_capacity;     /* blocks of it the device holds at once, at the current environments per warp */
  long long con_single_capacity;    /* ... and blocks (warps) of the single-warp constrained kernel */
  int *con_split_done;              /* device: FbParams::con_split_done */
  bool fast_block_auto;             /* 16 environments per warp chosen by the heuristic ... */
  int block_review;                 /* ... and reviewed after the first launch of an episode */
  int max_smem;
  long long launch_parity;
  int log_used;                     /* 0 until the first reset: the log is as fb_create zeroed it */
#ifndef FB_HOST_EMU
  FbFastEnvParams *fastQ;            /* host staging of the per-thread kernel's parameters (+ the ENVP twin's tables) */
  FbFastSplitEnvParams *splitQ;      /* ... of its SPLIT variant */
  FbFastConEnvParams *conQ;          /* ... and of the per-thread constrained kernel's */
  FbFastConSplitEnvParams *csplitQ;  /* ... and of its SPLIT variant */
#endif
  fbStream stream;
  std::vector<void *> allocs;
  int32_t *I_dev;
  float *F_dev;
  /* per-environment parameter tables (fb_set_env_param), indexed by FB_ENV_*: the device copy
   * (FbParams::ep_*, float32 [item*k + c][env_pad]) and the values as set ([n_envs][width]) */
  float *ep_dev[FB_N_ENV_PARAM];
  std::vector<double> ep_host[FB_N_ENV_PARAM];
  float *ep_lin;                    /* FbEnvTables::lin, derived while FB_ENV_ACT_BIAS is set (env_act_derive) */
  FbEnvTables ep;                   /* ep_dev and ep_lin as the kernels take it */
  /* per-environment episodes (fb_reset_envs): device [n_envs] batch iteration of each episode's row 0,
   * and whether one may be non-zero (a restart after iteration 0 since fb_reset) */
  long long *episode_start;
  bool episode_late;
  uint8_t *reset_mask;              /* fb_reset_envs staging (allocated at the first call): the mask ... */
  int *reset_list, *reset_row;      /* ... the uploaded list and each listed environment's row in it ... */
  float *reset_q, *reset_v;         /* ... and the uploaded rows [n][nq] / [n][nv] */
  long long launches;
  long long it;            /* batch iteration: physics steps since fb_reset */
  float last_ms;
  float *gather_links, *gather_joints;   /* fb_step_host staging */
  int joint_sel_n, joint_sel[32];        /* fb_set_host_joint_columns: columns of the joints row fb_step_host returns (0 = all) */
  int link_sel_n, link_sel[32];          /* fb_set_host_link_columns: the same for the links row */
  int link_items_n, link_items[64];      /* fb_set_host_link_items: links whose rows come down (0 = all) */
  int ctrl_sel_n, ctrl_sel[32];          /* fb_set_host_ctrl_columns: actuators fb_step_host's ctrl carries (0 = all nu) */
  float *export_stage[2];                /* fb_export_rows: dense row staging, double-buffered */
  size_t export_stage_floats;
  float *gather_env;                     /* fb_export_farms staging: one environment's ring of one kind */
  float *seq_dev, *seq_stage;            /* control sequence, environment-minor + upload staging */
  int seq_len, seq_pos, seq_cap, seq_rows;
  /* on-device CPG (fb_set_cpg): device tables + per-environment oscillator state */
  bool cpg_on;
  CpgDev cpg;
  std::vector<void *> cpg_allocs;
  float *cpg_theta0, *cpg_r0;          /* the state fb_set_cpg_state last set ([n_osc][env_pad]), for fb_reset_envs */
  std::vector<int> spring_qadr_host;   /* qpos addresses of the CPG's spring-reference outputs */
  const int *cpg_spring_qadr;          /* the same on the device */
  /* wave-controller copies (owned) */
  std::vector<int32_t> wc_act;
  std::vector<double> wc_amp, wc_freq, wc_lag, wc_off;
  bool has_wc;
  /* host copies of the user structs' arrays are not kept: hm holds the blobs */
  FbModel fm_shallow; FbFarms ff_shallow; bool has_farms;
  std::vector<std::vector<int32_t>> keep_i;
  std::vector<std::vector<double>> keep_d;
#ifndef FB_HOST_EMU
  cudaEvent_t ev0, ev1;
  cudaStream_t copy_stream;          /* device->host copies of fb_step_host_async */
  cudaStream_t gather_stream;        /* row gathers of fb_step_host (two buffer pairs: gathers of call i+1 overlap the copies of call i) */
  float *gather_links2, *gather_joints2;
  cudaStream_t up_stream;            /* ctrl upload of fb_step_host (SM reads of pinned host memory) */
  cudaEvent_t ev_up, ev_stage_free;
  float *ctrl_stage;                 /* [n_envs][nu] landing buffer of the upload, copied to ctrl in stream order */
  int sms;
  cudaEvent_t ev_gather, ev_gathered[4], ev_copy[4];  /* copy-done events of the last four pipelined calls (ring) */
  long long gather_it[4];            /* iteration whose ring row each of those calls gathers */
  long long host_calls;
#endif
};

template <typename Tp> static int alloc_arr(FbHandle *h, Tp **p, size_t count) {
  void *q = nullptr;
  if (dev_alloc(&q, count*sizeof(Tp))) return -1;
  h->allocs.push_back(q);
  *p = static_cast<Tp *>(q);
  return 0;
}

static const int32_t *keep_int(FbHandle *h, const int32_t *p, size_t n) {
  h->keep_i.emplace_back(p, p + n);
  if (h->keep_i.back().empty()) h->keep_i.back().push_back(0);
  return h->keep_i.back().data();
}
static const double *keep_dbl(FbHandle *h, const double *p, size_t n) {
  h->keep_d.emplace_back(p, p + n);
  if (h->keep_d.back().empty()) h->keep_d.back().push_back(0.0);
  return h->keep_d.back().data();
}

/* deep copies so that fb_set_wave_controller / fb_set_swimming can rebuild */
static void deep_copy_model(FbHandle *h, const FbModel *m, const FbFarms *f) {
  FbModel &d = h->fm_shallow;
  d = *m;
  const int nb = m->nbody, nj = m->njnt, nv = m->nv, nu = m->nu, ng = m->ngeom, nc = m->ncand;
#define KI(field, n) d.field = keep_int(h, m->field, (size_t)(n))
#define KD(field, n) d.field = keep_dbl(h, m->field, (size_t)(n))
  KI(body_parentid, nb); KI(body_jntid, nb); KI(body_dofadr, nb); KI(body_dofnum, nb);
  KD(body_pos, 3*nb); KD(body_quat, 4*nb); KD(body_ipos, 3*nb); KD(body_iquat, 4*nb);
  KD(body_mass, nb); KD(body_inertia, 3*nb); KD(body_invweight0, 2*nb);
  KI(jnt_type, nj); KI(jnt_bodyid, nj); KI(jnt_qposadr, nj); KI(jnt_dofadr, nj); KI(jnt_limited, nj);
  KD(jnt_pos, 3*nj); KD(jnt_axis, 3*nj); KD(jnt_stiffness, nj); KD(jnt_range, 2*nj);
  KD(jnt_margin, nj); KD(jnt_solref, 2*nj); KD(jnt_solimp, 5*nj);
  KI(dof_bodyid, nv); KI(dof_jntid, nv); KI(dof_parentid, nv); KI(dof_Madr, nv);
  KD(dof_damping, nv); KD(dof_armature, nv); KD(dof_invweight0, nv);
  KD(qpos0, m->nq); KD(qpos_spring, m->nq);
  KI(geom_type, ng); KI(geom_bodyid, ng); KD(geom_pos, 3*ng); KD(geom_quat, 4*ng); KD(geom_size, 3*ng);
  KI(cand_geom1, nc); KI(cand_geom2, nc); KI(cand_end, nc);
  KD(cand_friction, nc); KD(cand_solref, 2*nc); KD(cand_solimp, 5*nc); KD(cand_margin, nc); KD(cand_gap, nc);
  KI(actuator_trnid, nu); KI(actuator_ctrllimited, nu); KI(actuator_forcelimited, nu);
  KD(actuator_gainprm, 3*nu); KD(actuator_biasprm, 3*nu); KD(actuator_ctrlrange, 2*nu);
  KD(actuator_forcerange, 2*nu); KD(actuator_gear, nu);
  KD(key_qpos, m->nq); KD(key_qvel, nv);
#undef KI
#undef KD
  h->has_farms = f != nullptr;
  if (f) {
    FbFarms &e = h->ff_shallow;
    e = *f;
#define KI(field, n) e.field = keep_int(h, f->field, (size_t)(n))
#define KD(field, n) e.field = keep_dbl(h, f->field, (size_t)(n))
    KI(link_body, f->n_links); KI(joint_qposadr, f->n_joints); KI(joint_dofadr, f->n_joints);
    KI(joint_jntid, f->n_joints); KI(joint_act_position, f->n_joints);
    KI(joint_act_velocity, f->n_joints); KI(joint_act_torque, f->n_joints);
    KI(cand_sensor, 4*nc); KI(xfrc_body, f->n_xfrc);
    KI(swim_links_index, f->n_swim); KI(swim_xfrc_index, f->n_swim);
    KD(swim_mass, f->n_swim); KD(swim_height, f->n_swim); KD(swim_density, f->n_swim);
    KD(swim_coefficients, 6*f->n_swim);
#undef KI
#undef KD
  }
}

/* ---- per-environment parameters: the tables as the kernels take them */
static void env_param_bind(FbHandle *h) {
  h->ep.stiffness = h->ep_dev[FB_ENV_JNT_STIFFNESS];
  h->ep.damping = h->ep_dev[FB_ENV_DOF_DAMPING];
  h->ep.coef = h->ep_dev[FB_ENV_DRAG_COEF];
  h->ep.wvel = h->ep_dev[FB_ENV_WATER_VELOCITY];
  h->ep.fric = h->ep_dev[FB_ENV_CAND_FRICTION];
  h->ep.gain = h->ep_dev[FB_ENV_ACT_GAIN];
  h->ep.bias = h->ep_dev[FB_ENV_ACT_BIAS];
  h->ep.lin = h->ep_lin;
}

/* FbEnvTables::lin from the FB_ENV_ACT_BIAS table as set (double) and the current records: each
 * FT_ACT_SIMPLE joint's linear actuation form with environment e's biases, summed by the model
 * compiler's own fb_joint_actuation and rounded once, so that e steps bit for bit as a batch of the
 * model edited to its biases.  Freed while no bias table is set.  The gains feed no such sum: the
 * kernels read them from FB_ENV_ACT_GAIN where they use them. */
static int env_act_derive(FbHandle *h) {
  if (!h->ep_dev[FB_ENV_ACT_BIAS] || !h->hm.m.X.ok) {
    if (h->ep_lin) { dev_sync(h->stream); dev_free(h->ep_lin); h->ep_lin = nullptr; }
    env_param_bind(h);
    return 0;
  }
  const FbModel &fm = h->fm_shallow;
  const int n = h->P.n_envs, nu = fm.nu, nj = fm.njnt;
  const long long pad = h->P.env_pad;
  const int32_t *actwc = h->hm.I.data() + h->hm.m.o.ft_actwc;
  std::vector<float> dev((size_t)6*nj*pad, 0.f);
  for (size_t b = 1; b < h->hm.rec.size(); b++) {
    const FastRec &r = h->hm.rec[b];
    if (!(r.flags & FT_ACT_SIMPLE)) continue;
    for (int e = 0; e < n; e++) {
      const FbJointAct ja = fb_joint_actuation(&fm, h->has_farms ? &h->ff_shallow : nullptr, actwc, r,
                                               h->ep_host[FB_ENV_ACT_BIAS].data() + (size_t)e*3*nu, nullptr);
      const double t[6] = {ja.Kq, ja.Kqd, ja.T0, ja.KqU, ja.KqdU, ja.T0U};
      for (int k = 0; k < 6; k++) dev[(size_t)(6*r.jid + k)*pad + e] = (float)t[k];
    }
  }
  if (!h->ep_lin) {
    void *p = nullptr;
    if (dev_alloc(&p, dev.size()*sizeof(float))) return fail("per-environment actuator biases: device allocation failed");
    h->ep_lin = static_cast<float *>(p);
  }
  if (h2d(h->ep_lin, dev.data(), dev.size()*sizeof(float), h->stream) || dev_sync(h->stream))
    return fail(std::string("per-environment actuator biases: upload failed: ") + dev_error());
  env_param_bind(h);
  return 0;
}

/* (re)build the device model tables from the handle's host copies */
static int upload_model(FbHandle *h) {
  FbWaveController wc;
  wc.n = (int)h->wc_act.size();
  wc.actuator = h->wc_act.data(); wc.amplitude = h->wc_amp.data(); wc.frequency = h->wc_freq.data();
  wc.phase_lag = h->wc_lag.data(); wc.offset = h->wc_off.data();
  DevLayout keepL = h->hm.m.L;
  bool had = h->I_dev != nullptr;
  if (!fb_build_model(&h->fm_shallow, h->has_farms ? &h->ff_shallow : nullptr,
                      h->has_wc ? &wc : nullptr, h->team, h->hm))
    return fail("unsupported model: " + h->hm.error);
  if (had && memcmp(&keepL, &h->hm.m.L, sizeof(DevLayout)) != 0) return fail("layout changed on rebuild");
  if (h->I_dev) { dev_sync(h->stream); dev_free(h->I_dev); dev_free(h->F_dev); }
  void *pi = nullptr, *pf = nullptr;
  if (dev_alloc(&pi, h->hm.I.size()*sizeof(int32_t)) || dev_alloc(&pf, h->hm.F.size()*sizeof(float)))
    return fail("device allocation of the model tables failed");
  h->I_dev = static_cast<int32_t *>(pi);
  h->F_dev = static_cast<float *>(pf);
  if (h2d(h->I_dev, h->hm.I.data(), h->hm.I.size()*sizeof(int32_t), h->stream) ||
      h2d(h->F_dev, h->hm.F.data(), h->hm.F.size()*sizeof(float), h->stream) || dev_sync(h->stream))
    return fail("model upload failed");
  h->P.m = h->hm.m;
  h->P.m.I = h->I_dev;
  h->P.m.F = h->F_dev;
  /* spring-reference rows of the on-device CPG (the records were just rebuilt) */
  for (size_t sx = 0; sx < h->spring_qadr_host.size(); sx++)
    for (size_t b = 1; b < h->hm.rec.size(); b++)
      if (h->hm.rec[b].jtype >= 0 && h->hm.rec[b].jtype != FB_JNT_FREE && h->hm.rec[b].qa == h->spring_qadr_host[sx])
        h->hm.rec[b].flags |= (int32_t)(sx + 1) << FT_SREF_SHIFT;
#ifndef FB_HOST_EMU
  if (h->hm.m.X.ok) {
    if (!h->fastQ) h->fastQ = new FbFastEnvParams();
    memset(h->fastQ->rec, 0, sizeof(h->fastQ->rec));
    memcpy(h->fastQ->rec, h->hm.rec.data(), sizeof(FastRec)*h->hm.rec.size());
    if (!h->splitQ) h->splitQ = new FbFastSplitEnvParams();
    memcpy(h->splitQ->rec, h->fastQ->rec, sizeof(h->splitQ->rec));
    h->splitQ->split = h->hm.split;
    if (!h->conQ) h->conQ = new FbFastConEnvParams();
    memcpy(h->conQ->rec, h->fastQ->rec, sizeof(h->conQ->rec));
    memset(h->conQ->cand, 0, sizeof(h->conQ->cand));
    if (h->hm.m.X.con_ok) memcpy(h->conQ->cand, h->hm.crec.data(), sizeof(CandRec)*h->hm.crec.size());
    if (!h->csplitQ) h->csplitQ = new FbFastConSplitEnvParams();
    memcpy(h->csplitQ->rec, h->conQ->rec, sizeof(h->csplitQ->rec));
    memcpy(h->csplitQ->cand, h->conQ->cand, sizeof(h->csplitQ->cand));
    h->csplitQ->split = h->hm.split;
  }
#endif
  return env_act_derive(h);      /* the records' linear actuation forms may have changed */
}

/* capacity of the device control sequence ([n_steps][nu][env_pad] + the upload staging) */
static int ensure_sequence(FbHandle *h, int n_steps) {
  const DevModel &m = h->hm.m;
  const int rows = m.nu + h->cpg.n_spring;          /* ctrl rows + spring-reference rows per step */
  if (n_steps <= h->seq_cap && rows <= h->seq_rows) return 0;
  const size_t n = (size_t)h->P.n_envs, per_step = (size_t)rows*h->P.env_pad;
  h->seq_rows = rows;
  dev_sync(h->stream);
  if (h->seq_dev) { dev_free(h->seq_dev); dev_free(h->seq_stage); h->seq_dev = h->seq_stage = nullptr; h->seq_cap = 0; }
  void *a = nullptr, *b = nullptr;
  if (dev_alloc(&a, per_step*n_steps*sizeof(float)) || dev_alloc(&b, n*m.nu*n_steps*sizeof(float)))
    return fail("control sequence: device allocation failed");
  h->seq_dev = static_cast<float *>(a); h->seq_stage = static_cast<float *>(b);
  h->seq_cap = n_steps;
  return 0;
}

/* A per-thread kernel over the handle's batch with its launch shape: `blk` environments per warp
 * (per group for the constrained kernels), SLIM in blocks of `wpb` warps; LEAN and ENVP are 0. */
static FbKernelSel fb_kernel_sel(const FbHandle *h, int kind, int blk, int slim = 0, int wpb = 1) {
  const size_t per_env = (size_t)(slim ? h->hm.m.X.n_float_slim : h->hm.m.X.n_float)*sizeof(float);
  const int n = h->P.n_envs, warps = (n + 31)/32, split_threads = 32*h->hm.split.nwarps;
  FbKernelSel k = {kind, blk, slim, wpb > 1, 0, 0, (n + blk - 1)/blk, blk, per_env*blk};
  if (kind == FB_FAST_SPLIT) {
    k.grid = warps; k.threads = split_threads; k.bytes += FB_SPLIT_EXTRA_BYTES;
  } else if (kind == FB_FASTC_SPLIT) {
    k.threads = split_threads; k.bytes += (size_t)FB_CSPLIT_EXTRA*blk*sizeof(float);
  } else if (slim) {
    k.grid = (warps + wpb - 1)/wpb; k.threads = 32*wpb; k.bytes *= wpb;
  }
  return k;
}

#ifndef FB_HOST_EMU
/* blocks of `k` (any LEAN x ENVP) the device holds at once, its attributes set on the way; 0 on an error */
static long long fb_capacity(FbHandle *h, const FbKernelSel &k, cudaError_t *ce) {
  int per_sm = 0;
  if (*ce == cudaSuccess) *ce = fb_kernel_attributes(k, &per_sm);
  return *ce == cudaSuccess ? (long long)per_sm*h->sms : 0;
}

/* blocks of the constrained SPLIT variant the device holds at once with `blk` environments per group
 * (0: not applicable) */
static long long fb_con_split_blocks(FbHandle *h, int blk, cudaError_t *ce) {
  const FbKernelSel k = fb_kernel_sel(h, FB_FASTC_SPLIT, blk);
  if (!h->hm.m.X.con_ok || h->hm.split.nwarps < 2 || k.bytes > (size_t)h->max_smem) return 0;
  return fb_capacity(h, k, ce);
}

/* A ground-contact launch is as long as one group's step sequence times the number of waves its
 * blocks take: the SPLIT variant shortens the sequence (x FB_CSPLIT_GAIN, measured r2y: 1.7 .. 2.0
 * faster per wave) and holds fewer groups per wave.  Cost of stepping n_envs environments in
 * groups of blk, in units of a single-warp wave x 100; 0 = not available. */
#define FB_CSPLIT_GAIN 55
static long long fb_con_cost(long long n_envs, int blk, long long capacity, int split) {
  if (capacity <= 0) return 0;
  const long long groups = (n_envs + blk - 1)/blk, waves = (groups + capacity - 1)/capacity;
  return waves*(split ? FB_CSPLIT_GAIN : 100);
}
static bool fb_con_split_pays(const FbHandle *h) {
  const long long cs = fb_con_cost(h->P.n_envs, h->fast_block, h->con_split_capacity, 1);
  const long long c1 = fb_con_cost(h->P.n_envs, h->fast_block, h->con_single_capacity, 0);
  return cs > 0 && (c1 == 0 || cs < c1);
}

/* environments per warp of the per-thread kernels (regular layout): shared-memory attributes and
 * the capacities of the SPLIT variants and the single-warp constrained kernel */
static int fb_set_fast_block(FbHandle *h, int blk) {
  h->fast_block = blk;
  cudaError_t ce = fb_kernel_attributes(fb_kernel_sel(h, FB_FAST, blk));
  if (ce == cudaSuccess) ce = fb_kernel_attributes(fb_kernel_sel(h, FB_FASTC, blk));
  const FbKernelSel split = fb_kernel_sel(h, FB_FAST_SPLIT, 32), single = fb_kernel_sel(h, FB_FASTC, blk);
  /* the SPLIT variant pays while ALL its blocks are resident at once (one wave) */
  h->split_capacity = 0;
  if (blk == 32 && h->hm.split.nwarps > 1 && split.bytes <= (size_t)h->max_smem) h->split_capacity = fb_capacity(h, split, &ce);
  h->con_split_capacity = fb_con_split_blocks(h, blk, &ce);
  h->con_single_capacity = 0;
  if (h->hm.m.X.con_ok && single.bytes <= (size_t)h->max_smem) h->con_single_capacity = fb_capacity(h, single, &ce);
  return ce == cudaSuccess ? 0 : fail(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(ce));
}

/* shared-memory attributes of the SLIM variants (one warp per block, or 2..8 kept in step) */
static int fb_slim_attributes(FbHandle *h) {
  const FbKernelSel one = fb_kernel_sel(h, FB_FAST, 32, 1);
  int fit = h->max_smem/(int)one.bytes;     /* warps of one block that fit an SM's shared memory */
  if (fit > 8) fit = 8;
  FbKernelSel multi = fb_kernel_sel(h, FB_FAST, 32, 1, 2);
  multi.bytes = (fit >= 2 ? fit : 1)*one.bytes;
  cudaError_t ce = fb_kernel_attributes(one);
  if (ce == cudaSuccess) ce = fb_kernel_attributes(multi);
  if (ce != cudaSuccess) return fail(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(ce));
  if (h->fast_wpb > fit) h->fast_wpb = fit;
  if (h->fast_wpb < 2) h->fast_wpb = 1;
  return 0;
}
#endif

/* What one launch runs */
struct FbPlan {
  bool fast;            /* the unconstrained per-thread kernel `uncon` runs first; else the team kernel alone */
  FbKernelSel uncon;
  bool con_thread;      /* its hand-overs go to the per-thread constrained kernel `con`; else to the team kernel */
  bool con_split;       /* ... with the constrained SPLIT variant `csplit` launched in front */
  FbKernelSel con, csplit;
  int team_grid;        /* blocks of the team kernel (FbHandle::threads threads, smem_bytes bytes) */
};

/* The kernels a launch of `mode` runs.  The per-thread kernel advances every environment while it
 * is unconstrained; the constrained kernel or the team kernel finishes the ones it handed over.
 * Reset and derived-view requests go to the team kernel alone (it is the one that produces
 * mjData-like quantities).  The fb_* queries of the kernel selection read the plan of the next
 * fb_step. */
static FbPlan fb_plan(const FbHandle *h, int mode, int want_derived, bool ctrl_seq) {
  const DevModel &m = h->hm.m;
  const FbEnvTables &ep = h->ep;
  const int nw = h->hm.split.nwarps;
  FbPlan p = {};
  p.team_grid = (h->P.n_envs + h->envs_per_block - 1)/h->envs_per_block;
  p.fast = h->fast_enabled && m.X.ok && mode == FB_MODE_STEP && !want_derived;
  if (!p.fast) return p;
  /* LEAN: the same arithmetic with the model's unused paths compiled out; a control sequence needs
   * the general variant */
  const int lean = h->fast_lean && m.X.lean && !ctrl_seq;
  /* ENVP while a per-environment parameter table the kernel reads is set (the unconstrained kernels
   * never read the candidate friction), or the episode clock is bound: only while the wave
   * controller, the one step code that reads time, is on and some episode began after iteration 0 */
  const int envp = ep.stiffness || ep.damping || ep.coef || ep.wvel || ep.gain || ep.bias ||
                   (m.n_wc > 0 && h->episode_late);
  const int cenvp = envp || ep.fric;
#ifdef FB_HOST_EMU
  /* The emulation steps one environment at a time (BLK = 1; a constrained group is one
   * environment, so emu_per_thread gives the constrained SPLIT variant each handed-over environment
   * that has not stepped yet) and has no occupancy or cost model: the SPLIT variants run whenever
   * they are enabled and the model's tree splits. */
  const int blk = 1;
  const bool split = h->fast_split && !h->fast_slim && nw > 1;
  const bool con_split = h->con_split && !h->fast_slim && nw > 1;
#else
  const int blk = h->fast_block;
  const bool split = h->fast_split && !h->fast_slim && nw > 1 && blk == 32 && (h->P.n_envs + 31)/32 <= h->split_capacity;
  const bool con_split = h->con_split && !h->fast_slim && nw > 1 && fb_con_split_pays(h);
#endif
  if (split) {
    /* small batch: the tree of every 32 environments split over several warps */
    p.uncon = fb_kernel_sel(h, FB_FAST_SPLIT, blk);
  } else if (h->fast_slim && blk != 16) {
    /* multi-warp blocks: SLIM layout only (measured 3-5 % slower on the regular one) */
    p.uncon = fb_kernel_sel(h, FB_FAST, blk, 1, h->fast_wpb >= 2 && h->fast_wpb <= 8 ? h->fast_wpb : 1);
  } else {
    p.uncon = fb_kernel_sel(h, FB_FAST, blk);
  }
  p.uncon.lean = lean; p.uncon.envp = envp;
  p.con_thread = h->con_thread && m.X.con_ok;
  if (p.con_thread) {
    p.con = fb_kernel_sel(h, FB_FASTC, blk);
    p.con.lean = lean; p.con.envp = cenvp;
    /* small ground-contact batch: the tree of every group split over several warps */
    p.con_split = con_split;
    p.csplit = fb_kernel_sel(h, FB_FASTC_SPLIT, blk);
    p.csplit.lean = lean; p.csplit.envp = cenvp;
  }
  return p;
}

/* the plan of the next fb_step */
static FbPlan fb_next_step(const FbHandle *h) { return fb_plan(h, FB_MODE_STEP, 0, h->cpg_on || h->seq_len > 0); }

#ifdef FB_HOST_EMU
/* test harness: the warps of a SPLIT block as host threads meeting at FB_BLOCK_BARRIER */
template <class F> static void emu_split_run(int nw, F body) {
  pthread_barrier_t bar;
  pthread_barrier_init(&bar, nullptr, nw);
  fb_emu_bar = &bar;
  std::vector<std::thread> th;
  for (int r = 0; r < nw; r++) th.emplace_back(body, r);
  for (auto &t : th) t.join();
  fb_emu_bar = nullptr;
  pthread_barrier_destroy(&bar);
}

/* test harness: the body of the per-thread kernel `k` for one environment with BLK = 1; returns the
 * steps an unconstrained kernel completed */
static int emu_run(FbHandle *h, const FbParams &P, const FbKernelSel &k, int env, float *fs, float *fg, float *fc) {
  const FastSplit &sp = h->hm.split;
  const FastRec *rec = h->hm.rec.data();
  const CandRec *crec = h->hm.crec.data();
  int done = 0;
  fb_dispatch(k, [&](auto v) {
    using V = decltype(v);
    const FbEnvTables *T = V::envp ? &h->ep : nullptr;
    std::vector<float> extra(V::kind == FB_FAST_SPLIT || V::kind == FB_FASTC_SPLIT ? FB_CSPLIT_EXTRA : 0, 0.f);   /* one lane */
    if constexpr (V::kind == FB_FAST) {
      FbFast<1, V::slim, V::lean, 0, V::envp> st(P, rec, fs, fg, env, T);
      done = st.run(0, 0);
    } else if constexpr (V::kind == FB_FAST_SPLIT) {
      emu_split_run(sp.nwarps, [&](int role) {
        FbFast<1, 0, V::lean, 1, V::envp> st(P, rec, fs, fg, env, T);
        st.split_setup(sp, role, extra.data(), reinterpret_cast<int *>(extra.data() + 3));
        const int d = st.run_split(0, 0, 1);
        if (role == 0) done = d;
      });
    } else if constexpr (V::kind == FB_FASTC) {
      FbFastCon<1, V::lean, 0, V::envp> st(P, rec, crec, fs, fg, fc, env, T);
      st.run_con(P.steps_done[env], 0, 0);
    } else {
      emu_split_run(sp.nwarps, [&](int role) {
        FbFastCon<1, V::lean, 1, V::envp> st(P, rec, crec, fs, fg, fc, env, T);
        st.split_setup(sp, role, extra.data(), reinterpret_cast<int *>(extra.data() + 3));
        st.con_split_setup(sp, extra.data() + 4);
        st.run_con_split(0, 0);
      });
    }
  });
  return done;
}

/* test harness: the per-thread kernels of the plan run serially on the host */
static void emu_per_thread(FbHandle *h, FbParams &P, int n_steps, const FbPlan &plan) {
  const DevModel &m = P.m;
  P.pending_count[P.parity ^ 1] = 0;
  std::vector<float> fs((size_t)m.X.n_float + 8, 0.f);
  std::vector<float> fg((size_t)(m.X.n_scratch > m.X.n_scratch_slim ? m.X.n_scratch : m.X.n_scratch_slim) + 8, 0.f);
  std::vector<float> fc((size_t)m.X.n_con + 8, 0.f);
  for (int env = 0; env < P.n_envs; env++) {
    const int done = emu_run(h, P, plan.uncon, env, fs.data(), fg.data(), fc.data());
    if (done < n_steps) { P.steps_done[env] = done; P.pending[P.pending_count[P.parity]++] = env; }
  }
  if (!plan.con_thread) return;
  for (int i = 0; i < P.pending_count[P.parity]; i++) {
    const int env = P.pending[i];
    emu_run(h, P, plan.con_split && P.steps_done[env] == 0 ? plan.csplit : plan.con, env, fs.data(), fg.data(), fc.data());
  }
}
#else
template <class Q> static auto &fb_staging(FbHandle *h) {
  if constexpr (std::is_base_of_v<FbFastParams, Q>) return *h->fastQ;
  else if constexpr (std::is_base_of_v<FbFastSplitParams, Q>) return *h->splitQ;
  else if constexpr (std::is_base_of_v<FbFastConParams, Q>) return *h->conQ;
  else return *h->csplitQ;
}
template <class Q> static void fb_launch_kernel(FbHandle *h, const FbKernelSel &k, void (*kernel)(Q)) {
  auto &S = fb_staging<Q>(h);
  S.P = h->P; S.T = h->ep;
  kernel<<<k.grid, k.threads, k.bytes, h->stream>>>(static_cast<const Q &>(S));
}
/* launch the per-thread kernel `k` with the handle's parameters and tables */
static void fb_launch(FbHandle *h, const FbKernelSel &k) {
  fb_dispatch(k, [&](auto v) { fb_launch_kernel(h, k, fb_kernel_of(v)); });
  h->launches++;
}
#endif

/* only (FB_MODE_RESET): the environments fb_reset_envs restarts, at the current iteration; NULL: all */
static int launch(FbHandle *h, int mode, int n_steps, int want_derived, const uint8_t *only = nullptr) {
  FbParams &P = h->P;
  P.mode = mode; P.n_steps = n_steps; P.want_derived = want_derived; P.it0 = h->it;
  P.ctrl_seq = nullptr; P.seq_pos = 0;
  P.seq_stride = h->hm.m.nu; P.n_spring = 0; P.spring_qadr = nullptr;
  if (mode == FB_MODE_STEP && h->cpg_on) {
    if (ensure_sequence(h, n_steps)) return -1;
    const DevModel &dm = h->hm.m;
#ifdef FB_HOST_EMU
    for (int env = 0; env < P.n_envs; env++)
      fb_cpg_env(h->cpg, env, P.env_pad, n_steps, dm.nu, dm.timestep, P.ctrl, h->seq_dev);
#else
    fb_cpg_kernel<<<(P.n_envs + 127)/128, 128, 0, h->stream>>>(h->cpg, P.n_envs, P.env_pad, n_steps, dm.nu,
                                                                dm.timestep, P.ctrl, h->seq_dev);
    h->launches++;
#endif
    P.ctrl_seq = h->seq_dev; P.seq_pos = 0;
    P.n_spring = h->cpg.n_spring; P.seq_stride = dm.nu + h->cpg.n_spring; P.spring_qadr = h->cpg_spring_qadr;
  } else if (mode == FB_MODE_STEP && h->seq_len > 0) {
    if (h->seq_pos + n_steps > h->seq_len)
      return fail("fb_step: the control sequence holds fewer steps than requested");
    P.ctrl_seq = h->seq_dev; P.seq_pos = h->seq_pos;
    h->seq_pos += n_steps;
    if (h->seq_pos == h->seq_len) h->seq_len = h->seq_pos = 0;     /* consumed: ctrl is held again */
  }
  const FbPlan plan = fb_plan(h, mode, want_derived, P.ctrl_seq != nullptr);
  h->ep.episode_start = P.m.n_wc > 0 && h->episode_late ? h->episode_start : nullptr;
  P.use_pending = plan.fast;
  P.parity = (int)(h->launch_parity & 1);
  if (plan.fast) h->launch_parity++;
#ifdef FB_HOST_EMU
  const DevModel &m = P.m;
  if (plan.fast) emu_per_thread(h, P, n_steps, plan);
  std::vector<float> s((size_t)m.L.n_float + 8, 0.f);
  std::vector<int> si((size_t)m.L.n_int + 8, 0);
  const int count = plan.fast ? (plan.con_thread ? 0 : P.pending_count[P.parity]) : P.n_envs;
  for (int i = 0; i < count; i++) {
    int env = plan.fast ? P.pending[i] : i;
    if (only && !only[env]) continue;
    fb_run_env<1>(P, h->ep, env, plan.fast ? P.steps_done[env] : 0, s.data(), si.data(), 0, 0, 1u);
  }
  h->last_ms = 0.f;
  h->launches++;
#else
  if (h->host_calls > 0) {
    /* fb_step_host's row gathers run on the gather stream, in call order.  This launch overwrites
     * the ring rows of iterations it+1 .. it+n_steps, i.e. what iterations <= it+n_steps-ring left
     * there: it waits for the LATEST gather that reads such a row (row-less fb_step launches in
     * between count: the test is on iterations, not on this launch's length), which implies the
     * earlier ones.  Gathers older than the four tracked events are waited for through the oldest
     * tracked one; a reset waits for the latest. */
    long long dep = -1;
    const long long first = h->host_calls > 4 ? h->host_calls - 4 : 0;
    for (long long g = h->host_calls - 1; g >= first; g--)
      if (mode != FB_MODE_STEP || h->gather_it[g & 3] + P.ring <= h->it + n_steps) { dep = g; break; }
    if (dep < 0 && first > 0) dep = first;       /* long done in practice; covers calls before the window */
    if (dep >= 0 && cudaStreamWaitEvent(h->stream, h->ev_gathered[dep & 3], 0) != cudaSuccess) return fail(dev_error());
  }
  cudaEventRecord(h->ev0, h->stream);
  if (plan.fast) {
    fb_launch(h, plan.uncon);
    if (plan.con_thread) {
      P.con_split_done = plan.con_split ? h->con_split_done : nullptr;
      if (plan.con_split) fb_launch(h, plan.csplit);
      fb_launch(h, plan.con);
    }
  }
  if (!plan.con_thread) {
    fb_team_kernel(h->team)<<<plan.team_grid, h->threads, h->smem_bytes, h->stream>>>(P, h->ep, only);
    h->launches++;
  }
  cudaEventRecord(h->ev1, h->stream);
  {
    const cudaError_t le = cudaGetLastError();
    if (le != cudaSuccess) return fail(std::string("kernel launch failed: ") + cudaGetErrorString(le));
  }
#endif
  if (mode == FB_MODE_STEP) h->it += n_steps;       /* fb_reset set it to 0 before, fb_reset_envs keeps it */
#ifndef FB_HOST_EMU
  /* Half-filled warps (16 environments each) pay for candidate-rich models only through the
   * constrained step: a warp visits the union of its lanes' contacts.  Whether an episode is of
   * that kind shows in its first launch: when fewer than half of the environments were handed
   * over (a swimmer whose floor is far below), later launches use full warps, which is faster for
   * the unconstrained kernel at every batch size (r2l: 1.14e8 against 1.08e8 env-steps/s at 8,192
   * SALAMANDERs); ground-contact batches keep 16 (7.46e6 against 7.24e6 at 4,096).  The scratch
   * layouts depend on the block size but hold nothing across launches. */
  if (plan.fast && h->block_review) {
    h->block_review = 0;
    int both[2] = {0, 0};
    if (d2h(both, P.pending_count, sizeof(both), h->stream) || dev_sync(h->stream)) return fail(dev_error());
    int want = 2*both[P.parity] >= P.n_envs ? 16 : 32;
    if (want == 16 && plan.con_thread && h->con_split && h->hm.split.nwarps > 1) {
      /* with the constrained SPLIT variant a group is several warps: 16 per group pays only while
       * every group has an SM to itself (r2x, SALAMANDER ground: 1,024 envs 3.47e6 against 3.31e6
       * env-steps/s with 32; 4,096 envs 1.09e7 against 1.29e7); beyond that, whichever group size
       * needs fewer waves */
      cudaError_t ce = cudaSuccess;
      const long long c16 = fb_con_cost(P.n_envs, 16, fb_con_split_blocks(h, 16, &ce), 1);
      const long long c32 = fb_con_cost(P.n_envs, 32, fb_con_split_blocks(h, 32, &ce), 1);
      if (c32 > 0 && (c16 == 0 || c32 < c16 || (c32 == c16 && (P.n_envs + 15)/16 > h->sms))) want = 32;
    }
    if (want != h->fast_block && (size_t)P.m.X.n_float*sizeof(float)*want <= (size_t)h->max_smem && fb_set_fast_block(h, want)) return -1;
  }
#endif
  return 0;
}

#ifndef FB_HOST_EMU
/* FP32 roof of the device as this path could use it at best: every lane of every scheduler issuing
 * independent FFMAs from registers (8 chains per thread, 32 warps per SM).  bench.py quotes the
 * step kernels' arithmetic against this MEASURED figure (BASELINE.md section 2 asks the build for
 * it; the driver's MEASURED_PEAKS.json holds HBM and bf16 GEMM only). */
__global__ void __launch_bounds__(256) fb_ffma_peak_kernel(float *out, int iters, float a, float b) {
  float x0 = threadIdx.x*1e-3f, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f;
  float x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f, x7 = x0 + 7.f;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < 16; u++) {
      x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
      x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
  }
  const float r = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
  if (r == 123.456f) out[0] = r;       /* keeps the chains alive; never true for a = 1, b = 1e-9 */
}
#endif

template <typename Tsrc, typename Tdst>
static int cpg_upload(FbHandle *h, const Tsrc *src, size_t count, const Tdst **out) {
  std::vector<Tdst> tmp(count > 0 ? count : 1, Tdst(0));
  for (size_t i = 0; i < count; i++) tmp[i] = (Tdst)src[i];
  void *p = nullptr;
  if (dev_alloc(&p, tmp.size()*sizeof(Tdst))) return -1;
  h->cpg_allocs.push_back(p);
  if (h2d(p, tmp.data(), tmp.size()*sizeof(Tdst), h->stream) || dev_sync(h->stream)) return -1;
  *out = static_cast<const Tdst *>(p);
  return 0;
}

/* ------------------------------------------------------------------ ABI */
extern "C" {

const char *fb_last_error(void) { return g_error.c_str(); }
int fb_abi_version(void) { return FB_ABI_VERSION; }

void fb_destroy(FbHandle *h) {
  if (!h) return;
  dev_sync(h->stream);
  for (void *p : h->allocs) dev_free(p);
  for (int k = 0; k < 2; k++) if (h->export_stage[k]) dev_free(h->export_stage[k]);
  for (void *p : h->cpg_allocs) dev_free(p);
  if (h->seq_dev) { dev_free(h->seq_dev); dev_free(h->seq_stage); }
  if (h->I_dev) dev_free(h->I_dev);
  if (h->F_dev) dev_free(h->F_dev);
  for (float *p : h->ep_dev) if (p) dev_free(p);
  if (h->ep_lin) dev_free(h->ep_lin);
#ifndef FB_HOST_EMU
  cudaEventDestroy(h->ev0); cudaEventDestroy(h->ev1);
  cudaStreamSynchronize(h->copy_stream);
  cudaStreamSynchronize(h->up_stream);
  cudaStreamSynchronize(h->gather_stream);
  cudaStreamDestroy(h->gather_stream);
  cudaEventDestroy(h->ev_up); cudaEventDestroy(h->ev_stage_free);
  cudaStreamDestroy(h->up_stream);
  cudaEventDestroy(h->ev_gather);
  for (auto &e : h->ev_copy) cudaEventDestroy(e);
  for (auto &e : h->ev_gathered) cudaEventDestroy(e);
  cudaStreamDestroy(h->copy_stream);
  cudaStreamDestroy(h->stream);
  delete h->fastQ;
  delete h->conQ;
  delete h->splitQ;
  delete h->csplitQ;
#endif
  delete h;
}

int fb_create(const FbModel *model, const FbFarms *farms, int n_envs, int device, int ring_steps,
              int team_lanes, FbHandle **out) {
  if (!model || !out) return fail("fb_create: null argument");
  if (n_envs < 1 || ring_steps < 1) return fail("fb_create: n_envs and ring_steps must be >= 1");
  FbHandle *h = new (std::nothrow) FbHandle();
  if (!h) return fail("out of host memory");
  h->device = device; h->I_dev = nullptr; h->F_dev = nullptr; h->launches = 0; h->it = 0;
  for (float *&p : h->ep_dev) p = nullptr;
  h->ep_lin = nullptr;
  memset(&h->ep, 0, sizeof(h->ep));
  h->last_ms = 0.f; h->has_wc = false; h->gather_links = h->gather_joints = h->gather_env = nullptr;
  h->seq_dev = h->seq_stage = nullptr; h->seq_len = h->seq_pos = h->seq_cap = h->seq_rows = 0;
  h->cpg_on = false; memset(&h->cpg, 0, sizeof(h->cpg)); h->cpg_theta0 = h->cpg_r0 = nullptr;
  h->episode_start = nullptr; h->episode_late = false;
  h->reset_mask = nullptr; h->reset_list = h->reset_row = nullptr; h->reset_q = h->reset_v = nullptr;
  h->joint_sel_n = 0; h->link_sel_n = 0; h->link_items_n = 0; h->ctrl_sel_n = 0;
  h->export_stage[0] = h->export_stage[1] = nullptr; h->export_stage_floats = 0;
  h->fast_enabled = 1; h->fast_block = 1; h->launch_parity = 0;
  h->con_thread = 1; h->log_used = 0;
  if (const char *ev = getenv("FARMS_B200_CON_THREAD")) h->con_thread = atoi(ev) != 0;
  h->fast_slim = 0; h->fast_wpb = 1;
  h->fast_lean = 1; h->fast_block_auto = false; h->block_review = 0; h->max_smem = 0; h->fast_split = 0;
  h->split_capacity = 0; h->con_split = 0; h->con_split_capacity = 0; h->con_single_capacity = 0; h->con_split_done = nullptr;
  if (const char *ev = getenv("FARMS_B200_FAST_LEAN")) h->fast_lean = atoi(ev) != 0;
  if (const char *ev = getenv("FARMS_B200_FAST_SLIM")) h->fast_slim = atoi(ev) != 0;
#ifndef FB_HOST_EMU
  h->fastQ = nullptr; h->conQ = nullptr; h->splitQ = nullptr; h->csplitQ = nullptr;
#endif
  if (const char *ev = getenv("FARMS_B200_FAST")) h->fast_enabled = atoi(ev) != 0;
  memset(&h->P, 0, sizeof(h->P));
#ifdef FB_HOST_EMU
  h->stream = 0;
  h->team = 1;
  (void)team_lanes;
#else
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    delete h;
    return fail("no CUDA device: the engine has no CPU fallback");
  }
  if (device < 0 || device >= ndev) { delete h; return fail("fb_create: bad device index"); }
  cudaSetDevice(device);
  cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  cudaEventCreate(&h->ev0); cudaEventCreate(&h->ev1);
  {
    /* the row gathers must be dispatched while the next step kernel still has blocks waiting, so
     * their streams outrank it (measured: 3.3 ms behind the step kernel's second round, 0.13 ms
     * with priority).  The ctrl upload stays at normal priority: it is enqueued a launch ahead and
     * slips into the tail of the running step kernel; with priority it delays the first round of
     * the next one (e2e 2.67e8 -> 2.80e8 env-steps/s). */
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    cudaStreamCreateWithPriority(&h->copy_stream, cudaStreamNonBlocking, prio_hi);
    cudaStreamCreateWithPriority(&h->up_stream, cudaStreamNonBlocking, prio_lo);
    cudaStreamCreateWithPriority(&h->gather_stream, cudaStreamNonBlocking, prio_hi);
    h->gather_links2 = h->gather_joints2 = nullptr;
  }
  cudaEventCreateWithFlags(&h->ev_up, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&h->ev_stage_free, cudaEventDisableTiming);
  h->ctrl_stage = nullptr;
  h->sms = 148;
  cudaDeviceGetAttribute(&h->sms, cudaDevAttrMultiProcessorCount, device);
  cudaEventCreateWithFlags(&h->ev_gather, cudaEventDisableTiming);
  for (auto &e : h->ev_copy) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
  for (auto &e : h->ev_gathered) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
  h->host_calls = 0;
  for (auto &g : h->gather_it) g = 0;
  if (team_lanes != 0 && team_lanes != 8 && team_lanes != 16 && team_lanes != 32) {
    fb_destroy(h);
    return fail("fb_create: team_lanes must be 0, 8, 16 or 32");
  }
  h->team = team_lanes;
  if (h->team == 0) h->team = model->nbody > 20 ? 32 : (model->nbody > 10 ? 16 : 8);
  if (model->nbody > 2*h->team) {
    fb_destroy(h);
    return fail("fb_create: nbody exceeds 2*team_lanes (the subtree sums keep two bodies per lane in registers)");
  }
#endif
  deep_copy_model(h, model, farms);
  if (upload_model(h)) { fb_destroy(h); return -1; }
  const DevModel &m = h->hm.m;
#ifndef FB_HOST_EMU
  size_t per_env = (size_t)(m.L.n_float + m.L.n_int)*sizeof(float);
  int max_smem = 0;
  cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  if (per_env > (size_t)max_smem) { fb_destroy(h); return fail("model working set exceeds shared memory"); }
  int epb = 128/h->team;
  while (epb > 1 && per_env*epb > (size_t)max_smem/2) epb >>= 1;
  h->envs_per_block = epb;
  h->threads = epb*h->team;
  h->smem_bytes = per_env*epb;
  const cudaError_t ce = cudaFuncSetAttribute((const void *)fb_team_kernel(h->team), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_bytes);
  if (ce != cudaSuccess) { fb_destroy(h); return fail(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(ce)); }
  /* environment-per-thread kernels: one warp per block, as many blocks per SM as their
   * shared-memory working sets allow; models beyond that run on the team kernel.  A warp holds 32
   * environments.  Exception: a model with many collision candidates on a batch that leaves
   * schedulers idle anyway runs 16 per warp -- the constrained step visits the UNION of the
   * candidates its lanes touch and iterates until its slowest lane has converged, so half-filled
   * warps finish sooner (CENTIPEDE x 8,192: 60.5 -> 42.6 ms per 16 steps; slower everywhere else). */
  {
    size_t per_thread = (size_t)m.X.n_float*sizeof(float);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    h->fast_block = (m.ncand > 48 && n_envs/16 <= 4*sms) ? 16 : 32;
    if (const char *ev = getenv("FARMS_B200_FAST_BLOCK")) {
      const int v = atoi(ev);
      if (v == 16 || v == 32) h->fast_block = v;
    }
    h->fast_block_auto = getenv("FARMS_B200_FAST_BLOCK") == nullptr && h->fast_block == 16;
    h->max_smem = max_smem;
    if (!m.X.ok || per_thread*h->fast_block > (size_t)max_smem) h->fast_enabled = 0;
    if (h->fast_enabled) {
      if (fb_set_fast_block(h, h->fast_block)) { fb_destroy(h); return -1; }
      if (const char *ev = getenv("FARMS_B200_FAST_WPB")) h->fast_wpb = atoi(ev);

      /* SLIM layout: pays when the batch has more warps than the regular layout keeps resident
       * (4 per SM), i.e. when a second warp per scheduler exists to hide latencies behind */
      if (!getenv("FARMS_B200_FAST_SLIM"))
        h->fast_slim = h->fast_block == 32 && n_envs/32 > 4*sms && 8*per_thread*32 > (size_t)max_smem;   /* regular layout: < 8 warps per SM */
      if (h->fast_block != 32) h->fast_slim = 0;
      /* ... in blocks of up to 8 warps kept in step, one block per SM at a time: the launch takes
       * `rounds` blocks per SM one after the other, and the block size is the smallest that covers
       * the batch in that many rounds (65,536 environments on 148 SMs: 2 rounds of 7 warps, not
       * a round of 8 on every SM and a second one on 108 of them) */
      if (h->fast_slim && !getenv("FARMS_B200_FAST_WPB")) {
        const int warps = (n_envs + 31)/32, rounds = (warps + 8*sms - 1)/(8*sms);
        h->fast_wpb = (warps + sms*rounds - 1)/(sms*rounds);
        if (h->fast_wpb < 4) h->fast_wpb = 4;
      }
      if (h->fast_slim && fb_slim_attributes(h)) { fb_destroy(h); return -1; }
      /* SPLIT variant: pays while the batch leaves schedulers idle (a launch is then one warp's
       * latency, which the split shortens); beyond ~2 warps per scheduler the single-warp kernel
       * does the same work with fewer instructions */
      h->fast_split = !h->fast_slim && h->hm.split.nwarps > 1;     /* used while the batch fits one wave (launch) */
      if (const char *ev = getenv("FARMS_B200_FAST_SPLIT")) h->fast_split = atoi(ev) != 0;
      h->con_split = !h->fast_slim && h->hm.split.nwarps > 1 && m.X.con_ok;
      if (const char *ev = getenv("FARMS_B200_CON_SPLIT")) h->con_split = atoi(ev) != 0;
    }
  }
#else
  h->envs_per_block = 1; h->threads = 1;
  h->smem_bytes = (size_t)(m.L.n_float + m.L.n_int)*sizeof(float);
#endif
  FbParams &P = h->P;
  P.n_envs = n_envs; P.ring = ring_steps;
  const size_t n = (size_t)n_envs, nb = m.nbody, mc = m.maxcon > 0 ? m.maxcon : 1, nu = m.nu > 0 ? m.nu : 1;
  /* environment-minor log: rows of 32 consecutive environments are contiguous per vector */
  P.env_pad = (long long)((n_envs + 31) & ~31);
  int bad = 0;
  bad |= alloc_arr(h, &P.qpos, n*m.nq); bad |= alloc_arr(h, &P.qvel, n*m.nv);
  bad |= alloc_arr(h, &P.ctrl, n*nu); bad |= alloc_arr(h, &P.xfrc_applied, n*6*nb);
  bad |= alloc_arr(h, &P.qpos_spring, n*m.nq); bad |= alloc_arr(h, &P.env_phase, n);
  bad |= alloc_arr(h, &P.flags, n); bad |= alloc_arr(h, &P.iteration, n);
  bad |= alloc_arr(h, &P.pending, n); bad |= alloc_arr(h, &P.pending_count, 2); bad |= alloc_arr(h, &P.steps_done, n);
  bad |= alloc_arr(h, &P.con_dirty, n);
  bad |= alloc_arr(h, &h->episode_start, n);
  bad |= alloc_arr(h, &h->con_split_done, (n + 15)/16);
  P.fast_scratch_stride = (long long)((n + 31) & ~(size_t)31);
  P.fast_scratch = nullptr;
  if (m.X.ok) {
    const int ns = m.X.n_scratch > m.X.n_scratch_slim ? m.X.n_scratch : m.X.n_scratch_slim;
    bad |= alloc_arr(h, &P.fast_scratch, (size_t)P.fast_scratch_stride*(ns > 0 ? ns : 1));
  }
  P.con_scratch = nullptr;
  if (m.X.ok) bad |= alloc_arr(h, &P.con_scratch, (size_t)P.fast_scratch_stride*(m.X.n_con > 0 ? m.X.n_con : 1));
  bad |= alloc_arr(h, &P.d_xpos, n*3*nb); bad |= alloc_arr(h, &P.d_xquat, n*4*nb);
  bad |= alloc_arr(h, &P.d_xipos, n*3*nb); bad |= alloc_arr(h, &P.d_linvel, n*3*nb);
  bad |= alloc_arr(h, &P.d_angvel, n*3*nb); bad |= alloc_arr(h, &P.d_actf, n*nu);
  bad |= alloc_arr(h, &P.d_limf, n*(m.njnt > 0 ? m.njnt : 1)); bad |= alloc_arr(h, &P.d_qacc, n*m.nv);
  bad |= alloc_arr(h, &P.d_ncon, n); bad |= alloc_arr(h, &P.d_con_cand, n*mc);
  bad |= alloc_arr(h, &P.d_con_dist, n*mc); bad |= alloc_arr(h, &P.d_con_pos, n*3*mc);
  bad |= alloc_arr(h, &P.d_con_frame, n*9*mc); bad |= alloc_arr(h, &P.d_con_force, n*3*mc);
  bad |= alloc_arr(h, &P.J3, n*3*mc*m.nv); bad |= alloc_arr(h, &P.efc, n*5*(m.maxefc > 0 ? m.maxefc : 1));
  bad |= alloc_arr(h, &P.prod3, n*6*mc);
  const size_t ep = (size_t)P.env_pad*ring_steps;
  bad |= alloc_arr(h, &P.log_links, ep*m.n_links*20);
  bad |= alloc_arr(h, &P.log_joints, ep*m.n_joints*m.joint_cols);
  bad |= alloc_arr(h, &P.log_contacts, ep*m.n_contacts*12);
  bad |= alloc_arr(h, &P.log_xfrc, ep*m.n_xfrc*6);
  {
    size_t big = (size_t)ring_steps*m.n_links*20;
    if ((size_t)ring_steps*m.n_joints*m.joint_cols > big) big = (size_t)ring_steps*m.n_joints*m.joint_cols;
    if ((size_t)ring_steps*m.n_contacts*12 > big) big = (size_t)ring_steps*m.n_contacts*12;
    if ((size_t)ring_steps*m.n_xfrc*6 > big) big = (size_t)ring_steps*m.n_xfrc*6;
    bad |= alloc_arr(h, &h->gather_env, big > 0 ? big : 1);
  }
  bad |= alloc_arr(h, &h->gather_links, n*m.n_links*20);
  bad |= alloc_arr(h, &h->gather_joints, n*m.n_joints*m.joint_cols);
  if (bad) { fb_destroy(h); return fail("device allocation failed (n_envs x ring too large?)"); }
  /* qpos_spring <- model value for every environment */
  std::vector<float> spring((size_t)n*m.nq);
  for (size_t e = 0; e < n; e++)
    for (int i = 0; i < m.nq; i++) spring[e*m.nq + i] = (float)model->qpos_spring[i];
  if (h2d(P.qpos_spring, spring.data(), spring.size()*sizeof(float), h->stream) || dev_sync(h->stream)) {
    fb_destroy(h);
    return fail("upload failed");
  }
  *out = h;
  return fb_reset(h, nullptr, nullptr);
}

int fb_reset(FbHandle *h, const double *qpos0, const double *qvel0) {
  if (!h) return fail("null handle");
  const DevModel &m = h->hm.m;
  const size_t n = (size_t)h->P.n_envs;
  std::vector<float> q(n*m.nq), v(n*m.nv);
  for (size_t e = 0; e < n; e++) {
    for (int i = 0; i < m.nq; i++)
      q[e*m.nq + i] = qpos0 ? (float)qpos0[e*m.nq + i] : h->hm.F[h->hm.m.o.key_qpos + i];
    for (int i = 0; i < m.nv; i++)
      v[e*m.nv + i] = qvel0 ? (float)qvel0[e*m.nv + i] : h->hm.F[h->hm.m.o.key_qvel + i];
  }
  FbParams &P = h->P;
  /* The unconstrained kernel relies on a log whose constraint-only columns start as zeros
   * (FbParams::con_dirty): fresh from fb_create they are; a later reset clears what the previous
   * episode left in the contacts and joints rows. */
  std::vector<long long> never(n, FB_NEVER_DIRTY);
  int bad = h2d(P.con_dirty, never.data(), n*sizeof(long long), h->stream);
  if (h->log_used) {
    const size_t ep = (size_t)P.env_pad*P.ring;
    bad |= dev_zero(P.log_contacts, ep*m.n_contacts*12*sizeof(float), h->stream);
    bad |= dev_zero(P.log_joints, ep*m.n_joints*m.joint_cols*sizeof(float), h->stream);
  }
  h->log_used = 1;
  bad |= h2d(P.qpos, q.data(), q.size()*sizeof(float), h->stream);
  bad |= h2d(P.qvel, v.data(), v.size()*sizeof(float), h->stream);
  bad |= dev_zero(P.ctrl, n*(m.nu > 0 ? m.nu : 1)*sizeof(float), h->stream);
  bad |= dev_zero(P.xfrc_applied, n*6*m.nbody*sizeof(float), h->stream);
  bad |= dev_zero(P.flags, n*sizeof(int), h->stream);
  bad |= dev_zero(h->episode_start, n*sizeof(long long), h->stream);
  bad |= dev_sync(h->stream);   /* q, v are stack-owned */
  if (bad) return fail(std::string("fb_reset: ") + dev_error());
  h->it = 0;
  h->episode_late = false;
  h->seq_len = h->seq_pos = 0;
#ifndef FB_HOST_EMU
  if (h->fast_enabled && h->fast_block_auto) {
    if (h->fast_block != 16 && fb_set_fast_block(h, 16)) return -1;
    h->block_review = 1;
  }
#endif
  if (launch(h, FB_MODE_RESET, 1, 1)) return -1;
  return dev_sync(h->stream) ? fail(std::string("fb_reset: ") + dev_error()) : 0;
}

/* fb_reset_envs / fb_reset_envs_where: the state rows, CPG rows and episode start of the masked
 * environments, then the reset's forward pass for them alone (log row it % ring, derived view), all
 * on the handle's stream and without a host synchronisation */
static int reset_envs_enqueue(FbHandle *h, const uint8_t *mask, const int *row_of, const float *qpos0, const float *qvel0) {
  FbParams &P = h->P;
  const DevModel &m = h->hm.m;
  FbResetArgs A;
  A.mask = mask; A.qpos0 = qpos0; A.qvel0 = qvel0; A.row_of = row_of;
  A.key_qpos = h->F_dev + m.o.key_qpos; A.key_qvel = h->F_dev + m.o.key_qvel;
  A.qpos = P.qpos; A.qvel = P.qvel; A.ctrl = P.ctrl; A.xfrc_applied = P.xfrc_applied; A.flags = P.flags;
  A.episode_start = h->episode_start;
  A.n_osc = h->cpg_on ? h->cpg.n_osc : 0;
  A.theta = h->cpg.theta; A.r = h->cpg.r; A.rd = h->cpg.rd; A.theta0 = h->cpg_theta0; A.r0 = h->cpg_r0;
  A.n_envs = P.n_envs; A.nq = m.nq; A.nv = m.nv; A.nu = m.nu; A.nbody = m.nbody;
  A.env_pad = P.env_pad; A.it = h->it;
#ifdef FB_HOST_EMU
  for (int env = 0; env < P.n_envs; env++) fb_reset_env(A, env);
#else
  fb_reset_envs_kernel<<<(P.n_envs + 127)/128, 128, 0, h->stream>>>(A);
  h->launches++;
#endif
  if (h->it > 0) h->episode_late = true;
  return launch(h, FB_MODE_RESET, 1, 1, mask);
}

int fb_reset_envs(FbHandle *h, int n, const int32_t *envs, const double *qpos0, const double *qvel0) {
  if (!h) return fail("null handle");
  if (n < 0 || (n > 0 && !envs)) return fail("fb_reset_envs: n must be >= 0, with envs[n]");
  if (n == 0) return 0;
  const DevModel &m = h->hm.m;
  const int N = h->P.n_envs;
  std::vector<int> seen((size_t)N, -1);
  for (int i = 0; i < n; i++) {
    const int e = envs[i];
    if (e < 0 || e >= N)
      return fail("fb_reset_envs: envs[" + std::to_string(i) + "] = " + std::to_string(e) + " is out of range [0, " +
                  std::to_string(N) + ")");
    if (seen[e] >= 0)
      return fail("fb_reset_envs: environment " + std::to_string(e) + " is given twice (envs[" + std::to_string(seen[e]) +
                  "] and envs[" + std::to_string(i) + "])");
    seen[e] = i;
  }
  std::vector<float> q(qpos0 ? (size_t)n*m.nq : 0), v(qvel0 ? (size_t)n*m.nv : 0);
  const struct { const double *src; std::vector<float> &dst; int w; const char *name; } rows[2] = {
    {qpos0, q, m.nq, "qpos0"}, {qvel0, v, m.nv, "qvel0"}};
  for (const auto &r : rows)
    for (size_t k = 0; k < r.dst.size(); k++) {
      if (!std::isfinite(r.src[k]))
        return fail(std::string("fb_reset_envs: non-finite ") + r.name + " at row " + std::to_string(k/r.w) +
                    " (environment " + std::to_string(envs[k/r.w]) + "), index " + std::to_string(k % r.w));
      r.dst[k] = (float)r.src[k];
    }
  if (!h->reset_mask) {
    int bad = alloc_arr(h, &h->reset_mask, (size_t)N);
    bad |= alloc_arr(h, &h->reset_list, (size_t)N); bad |= alloc_arr(h, &h->reset_row, (size_t)N);
    bad |= alloc_arr(h, &h->reset_q, (size_t)N*m.nq); bad |= alloc_arr(h, &h->reset_v, (size_t)N*m.nv);
    if (bad) return fail("fb_reset_envs: device allocation failed");
  }
  int bad = dev_zero(h->reset_mask, (size_t)N, h->stream);
  bad |= h2d(h->reset_list, envs, (size_t)n*sizeof(int32_t), h->stream);
  if (qpos0) bad |= h2d(h->reset_q, q.data(), q.size()*sizeof(float), h->stream);
  if (qvel0) bad |= h2d(h->reset_v, v.data(), v.size()*sizeof(float), h->stream);
  if (bad) return fail(std::string("fb_reset_envs: ") + dev_error());
#ifdef FB_HOST_EMU
  for (int i = 0; i < n; i++) { h->reset_mask[envs[i]] = 1; h->reset_row[envs[i]] = i; }
#else
  fb_reset_list_kernel<<<(n + 127)/128, 128, 0, h->stream>>>(h->reset_list, n, h->reset_mask, h->reset_row);
  h->launches++;
#endif
  if (reset_envs_enqueue(h, h->reset_mask, h->reset_row, qpos0 ? h->reset_q : nullptr, qvel0 ? h->reset_v : nullptr))
    return -1;
  return dev_sync(h->stream) ? fail(std::string("fb_reset_envs: ") + dev_error()) : 0;   /* q, v are stack-owned */
}

int fb_reset_envs_where(FbHandle *h, const uint8_t *mask, const float *qpos0, const float *qvel0) {
  if (!h) return fail("null handle");
  if (!mask) return fail("fb_reset_envs_where: null mask");
  return reset_envs_enqueue(h, mask, nullptr, qpos0, qvel0);
}

int fb_get_episode_start(FbHandle *h, int64_t *out) {
  if (!h || !out) return fail("null argument");
  if (d2h(out, h->episode_start, (size_t)h->P.n_envs*sizeof(long long), h->stream) || dev_sync(h->stream))
    return fail(std::string("fb_get_episode_start: ") + dev_error());
  return 0;
}

static int upload_doubles(FbHandle *h, float *dst, const double *src, size_t count, const char *what) {
  if (!h || !src) return fail(std::string(what) + ": null argument");
  std::vector<float> tmp(count);
  for (size_t i = 0; i < count; i++) tmp[i] = (float)src[i];
  if (h2d(dst, tmp.data(), count*sizeof(float), h->stream) || dev_sync(h->stream))
    return fail(std::string(what) + ": " + dev_error());
  return 0;
}

int fb_set_ctrl(FbHandle *h, const double *ctrl) {
  return upload_doubles(h, h->P.ctrl, ctrl, (size_t)h->P.n_envs*h->hm.m.nu, "fb_set_ctrl");
}
int fb_set_ctrl_sequence(FbHandle *h, const float *ctrl, int n_steps) {
  if (!h) return fail("null handle");
  h->seq_len = h->seq_pos = 0;
  if (!ctrl || n_steps <= 0) return 0;              /* sequence off */
  const DevModel &m = h->hm.m;
  if (m.nu <= 0) return fail("fb_set_ctrl_sequence: the model has no actuators");
  if (h->cpg_on) return fail("fb_set_ctrl_sequence: the on-device CPG owns the control sequence (fb_set_cpg(h, NULL) first)");
  const size_t n = (size_t)h->P.n_envs;
  if (ensure_sequence(h, n_steps)) return -1;
#ifdef FB_HOST_EMU
  for (int k = 0; k < n_steps; k++)
    for (size_t e = 0; e < n; e++)
      for (int a = 0; a < m.nu; a++)
        h->seq_dev[((size_t)k*m.nu + a)*h->P.env_pad + e] = ctrl[((size_t)k*n + e)*m.nu + a];
#else
  if (h2d(h->seq_stage, ctrl, n*m.nu*n_steps*sizeof(float), h->stream)) return fail(dev_error());
  long long total = (long long)n_steps*m.nu*(long long)n;
  fb_transpose_ctrl_kernel<<<(unsigned)((total + 255)/256), 256, 0, h->stream>>>(
      h->seq_stage, n_steps, (int)n, m.nu, h->P.env_pad, h->seq_dev);
  h->launches++;
  if (dev_sync(h->stream)) return fail(std::string("fb_set_ctrl_sequence: ") + dev_error());   /* ctrl is the caller's */
#endif
  h->seq_len = n_steps;
  return 0;
}

int fb_set_qpos_spring(FbHandle *h, const double *qs) {
  return upload_doubles(h, h->P.qpos_spring, qs, (size_t)h->P.n_envs*h->hm.m.nq, "fb_set_qpos_spring");
}
int fb_set_env_phase(FbHandle *h, const double *phase) {
  return upload_doubles(h, h->P.env_phase, phase, (size_t)h->P.n_envs, "fb_set_env_phase");
}

int fb_set_wave_controller(FbHandle *h, const FbWaveController *c) {
  if (!h) return fail("null handle");
  h->has_wc = c != nullptr && c->n > 0;
  h->wc_act.clear(); h->wc_amp.clear(); h->wc_freq.clear(); h->wc_lag.clear(); h->wc_off.clear();
  if (h->has_wc) {
    for (int i = 0; i < c->n; i++) {
      if (c->actuator[i] < 0 || c->actuator[i] >= h->hm.m.nu) return fail("wave controller: bad actuator index");
      h->wc_act.push_back(c->actuator[i]);
      h->wc_amp.push_back(c->amplitude[i]); h->wc_freq.push_back(c->frequency[i]);
      h->wc_lag.push_back(c->phase_lag[i]); h->wc_off.push_back(c->offset ? c->offset[i] : 0.0);
    }
  }
  return upload_model(h);
}

int fb_set_cpg(FbHandle *h, const FbCpgNetwork *net) {
  if (!h) return fail("null handle");
  dev_sync(h->stream);
  for (void *p : h->cpg_allocs) dev_free(p);
  h->cpg_allocs.clear();
  h->cpg_on = false;
  memset(&h->cpg, 0, sizeof(h->cpg));
  h->cpg_theta0 = h->cpg_r0 = nullptr;
  h->cpg_spring_qadr = nullptr;
  if (!h->spring_qadr_host.empty()) {
    h->spring_qadr_host.clear();
    if (upload_model(h)) return -1;              /* records without spring rows */
  }
  if (!net || net->n_osc <= 0) return 0;
  const DevModel &m = h->hm.m;
  if (net->n_osc > FB_CPG_MAXOSC) return fail("fb_set_cpg: at most 64 oscillators");
  if (m.nu <= 0) return fail("fb_set_cpg: the model has no actuators");
  for (int e = 0; e < net->n_coupling; e++)
    if (net->coupling_from[e] < 0 || net->coupling_from[e] >= net->n_osc || net->coupling_to[e] < 0 ||
        net->coupling_to[e] >= net->n_osc) return fail("fb_set_cpg: coupling index out of range");
  for (int o = 0; o < net->n_out; o++)
    if (net->out_actuator[o] < 0 || net->out_actuator[o] >= m.nu || net->out_osc_a[o] < 0 ||
        net->out_osc_a[o] >= net->n_osc || net->out_osc_b[o] >= net->n_osc)
      return fail("fb_set_cpg: output index out of range");
  CpgDev &c = h->cpg;
  c.n_osc = net->n_osc; c.n_coupling = net->n_coupling; c.n_out = net->n_out;
  int bad = 0;
  bad |= cpg_upload(h, net->frequency, net->n_osc, &c.freq);
  bad |= cpg_upload(h, net->amplitude, net->n_osc, &c.amp);
  bad |= cpg_upload(h, net->rate, net->n_osc, &c.rate);
  bad |= cpg_upload(h, net->coupling_from, net->n_coupling, &c.c_from);
  bad |= cpg_upload(h, net->coupling_to, net->n_coupling, &c.c_to);
  bad |= cpg_upload(h, net->coupling_weight, net->n_coupling, &c.c_w);
  bad |= cpg_upload(h, net->coupling_bias, net->n_coupling, &c.c_phi);
  bad |= cpg_upload(h, net->out_actuator, net->n_out, &c.o_act);
  bad |= cpg_upload(h, net->out_osc_a, net->n_out, &c.o_a);
  bad |= cpg_upload(h, net->out_osc_b, net->n_out, &c.o_b);
  bad |= cpg_upload(h, net->out_gain, net->n_out, &c.o_gain);
  bad |= cpg_upload(h, net->out_offset, net->n_out, &c.o_off);
  const size_t st = (size_t)net->n_osc*h->P.env_pad;
  void *pt = nullptr, *pr = nullptr, *pd = nullptr, *pt0 = nullptr, *pr0 = nullptr;
  bad |= dev_alloc(&pt, st*sizeof(float)); bad |= dev_alloc(&pr, st*sizeof(float)); bad |= dev_alloc(&pd, st*sizeof(float));
  bad |= dev_alloc(&pt0, st*sizeof(float)); bad |= dev_alloc(&pr0, st*sizeof(float));
  if (bad) return fail("fb_set_cpg: device allocation / upload failed");
  for (void *p : {pt, pr, pd, pt0, pr0}) h->cpg_allocs.push_back(p);
  c.theta = static_cast<float *>(pt); c.r = static_cast<float *>(pr); c.rd = static_cast<float *>(pd);
  h->cpg_theta0 = static_cast<float *>(pt0); h->cpg_r0 = static_cast<float *>(pr0);
  h->cpg_on = true;
  h->seq_len = h->seq_pos = 0;
  return 0;
}

int fb_set_cpg_springrefs(FbHandle *h, int n, const int32_t *qpos_adr, const int32_t *osc_a, const int32_t *osc_b,
                          const double *gain, const double *offset) {
  if (!h) return fail("null handle");
  if (!h->cpg_on) return fail("fb_set_cpg_springrefs: no CPG set (fb_set_cpg first)");
  if (n < 0 || (n > 0 && (!qpos_adr || !osc_a || !osc_b || !gain || !offset))) return fail("fb_set_cpg_springrefs: null argument");
  if (n > FB_MAX_SPRINGREFS) return fail("fb_set_cpg_springrefs: at most 126 spring references");
  dev_sync(h->stream);
  const DevModel &m = h->hm.m;
  std::vector<int> adr;
  for (int i = 0; i < n; i++) {
    if (osc_a[i] < 0 || osc_a[i] >= h->cpg.n_osc || osc_b[i] >= h->cpg.n_osc) return fail("fb_set_cpg_springrefs: oscillator index out of range");
    bool found = false;
    for (int j = 0; j < m.njnt && !found; j++)
      found = h->hm.I[m.o.jnt_qposadr + j] == qpos_adr[i] && h->hm.I[m.o.jnt_type + j] != FB_JNT_FREE;
    if (!found) return fail("fb_set_cpg_springrefs: not the qpos address of a hinge or slide joint");
    for (int k : adr) if (k == qpos_adr[i]) return fail("fb_set_cpg_springrefs: a joint is listed twice");
    adr.push_back(qpos_adr[i]);
  }
  CpgDev &c = h->cpg;
  c.n_spring = 0;
  h->spring_qadr_host = adr;
  if (upload_model(h)) return -1;                /* rebuilds the records with their spring rows */
  if (n == 0) return 0;
  int bad = 0;
  bad |= cpg_upload(h, osc_a, n, &c.s_a);
  bad |= cpg_upload(h, osc_b, n, &c.s_b);
  bad |= cpg_upload(h, gain, n, &c.s_gain);
  bad |= cpg_upload(h, offset, n, &c.s_off);
  bad |= cpg_upload(h, adr.data(), n, &h->cpg_spring_qadr);
  if (bad) return fail("fb_set_cpg_springrefs: device allocation / upload failed");
  c.n_spring = n;
  return 0;
}

int fb_set_cpg_state(FbHandle *h, const double *phase, const double *amplitude) {
  if (!h || !phase) return fail("null argument");
  if (!h->cpg_on) return fail("fb_set_cpg_state: no CPG set");
  const size_t n = (size_t)h->P.n_envs, pad = (size_t)h->P.env_pad, no = (size_t)h->cpg.n_osc;
  std::vector<float> th(no*pad, 0.f), r(no*pad, 0.f), rd(no*pad, 0.f);
  for (size_t e = 0; e < n; e++)
    for (size_t i = 0; i < no; i++) {
      th[i*pad + e] = (float)phase[e*no + i];
      if (amplitude) r[i*pad + e] = (float)amplitude[e*no + i];
    }
  /* the device copy in cpg_theta0 / cpg_r0 is what fb_reset_envs restores */
  if (h2d(h->cpg.theta, th.data(), th.size()*sizeof(float), h->stream) ||
      h2d(h->cpg.r, r.data(), r.size()*sizeof(float), h->stream) ||
      h2d(h->cpg.rd, rd.data(), rd.size()*sizeof(float), h->stream) ||
      h2d(h->cpg_theta0, th.data(), th.size()*sizeof(float), h->stream) ||
      h2d(h->cpg_r0, r.data(), r.size()*sizeof(float), h->stream) || dev_sync(h->stream))
    return fail(std::string("fb_set_cpg_state: ") + dev_error());
  return 0;
}

int fb_get_cpg_state(FbHandle *h, double *phase, double *amplitude) {
  if (!h || !phase) return fail("null argument");
  if (!h->cpg_on) return fail("fb_get_cpg_state: no CPG set");
  const size_t n = (size_t)h->P.n_envs, pad = (size_t)h->P.env_pad, no = (size_t)h->cpg.n_osc;
  std::vector<float> th(no*pad), r(no*pad);
  if (d2h(th.data(), h->cpg.theta, th.size()*sizeof(float), h->stream) ||
      d2h(r.data(), h->cpg.r, r.size()*sizeof(float), h->stream) || dev_sync(h->stream))
    return fail(std::string("fb_get_cpg_state: ") + dev_error());
  for (size_t e = 0; e < n; e++)
    for (size_t i = 0; i < no; i++) {
      phase[e*no + i] = th[i*pad + e];
      if (amplitude) amplitude[e*no + i] = r[i*pad + e];
    }
  return 0;
}

int fb_set_actuator_forcerange(FbHandle *h, int n, const int32_t *actuator, const int32_t *limited,
                               const double *range) {
  if (!h || (n > 0 && (!actuator || !limited || !range))) return fail("null argument");
  /* the handle owns deep copies of the model arrays (deep_copy_model): edit them, rebuild */
  int32_t *fl = const_cast<int32_t *>(h->fm_shallow.actuator_forcelimited);
  double *fr = const_cast<double *>(h->fm_shallow.actuator_forcerange);
  for (int i = 0; i < n; i++) {
    int a = actuator[i];
    if (a < 0 || a >= h->fm_shallow.nu) return fail("fb_set_actuator_forcerange: bad actuator index");
    fl[a] = limited[i] != 0;
    fr[2*a] = range[2*i]; fr[2*a + 1] = range[2*i + 1];
  }
  return upload_model(h);
}

int fb_set_water_velocity(FbHandle *h, double vx, double vy, double vz) {
  if (!h) return fail("null handle");
  if (!h->has_farms) return fail("no farms tables");
  if (h->ep_dev[FB_ENV_WATER_VELOCITY])
    return fail("fb_set_water_velocity: a per-environment water velocity is set; change it with "
                "fb_set_env_param(FB_ENV_WATER_VELOCITY, ...), or clear it with fb_set_env_param(FB_ENV_WATER_VELOCITY, NULL) first");
  h->ff_shallow.water_velocity[0] = vx; h->ff_shallow.water_velocity[1] = vy; h->ff_shallow.water_velocity[2] = vz;
  h->P.m.water_velocity[0] = (float)vx; h->P.m.water_velocity[1] = (float)vy; h->P.m.water_velocity[2] = (float)vz;
  h->hm.m.water_velocity[0] = (float)vx; h->hm.m.water_velocity[1] = (float)vy; h->hm.m.water_velocity[2] = (float)vz;
  return 0;
}

/* ---- per-environment parameters (fb_set_env_param) */
static const char *const kEnvParamName[FB_N_ENV_PARAM] = {"FB_ENV_JNT_STIFFNESS", "FB_ENV_DOF_DAMPING", "FB_ENV_DRAG_COEF",
                                                          "FB_ENV_WATER_VELOCITY", "FB_ENV_CAND_FRICTION",
                                                          "FB_ENV_ACT_GAIN", "FB_ENV_ACT_BIAS"};

/* Lowest candidate friction a table may hold (mjcf_subset.PAIR_MIN_FRICTION): the pyramid rows'
 * D = 1/(2 mu^2 R) stiffens as 1/mu^2, and the fp32 solver's error grows with it (DESIGN.md section 8) */
#define FB_MIN_ENV_FRICTION 0.1

/* values per environment of a field: njnt, nv, 6*n_swim, 3, ncand, nu, 3*nu */
static int env_param_width(const FbHandle *h, int field) {
  switch (field) {
    case FB_ENV_ACT_GAIN: return h->fm_shallow.nu;
    case FB_ENV_ACT_BIAS: return 3*h->fm_shallow.nu;
    case FB_ENV_JNT_STIFFNESS: return h->fm_shallow.njnt;
    case FB_ENV_DOF_DAMPING: return h->fm_shallow.nv;
    case FB_ENV_DRAG_COEF: return h->has_farms ? 6*h->ff_shallow.n_swim : 0;
    case FB_ENV_CAND_FRICTION: return h->fm_shallow.ncand;
    default: return 3;
  }
}

/* the model's value of entry c of a field */
static double env_param_model(const FbHandle *h, int field, int c) {
  switch (field) {
    case FB_ENV_JNT_STIFFNESS: return h->fm_shallow.jnt_stiffness[c];
    case FB_ENV_DOF_DAMPING: return h->fm_shallow.dof_damping[c];
    case FB_ENV_DRAG_COEF: return h->ff_shallow.swim_coefficients[c];
    case FB_ENV_CAND_FRICTION: return h->fm_shallow.cand_friction[c];
    case FB_ENV_ACT_GAIN: return h->fm_shallow.actuator_gainprm[3*c];
    case FB_ENV_ACT_BIAS: return h->fm_shallow.actuator_biasprm[c];
    default: return h->has_farms ? h->ff_shallow.water_velocity[c] : 0.0;
  }
}

int fb_set_env_param(FbHandle *h, int field, const double *values) {
  if (!h) return fail("null handle");
  if (field < 0 || field >= FB_N_ENV_PARAM) return fail("fb_set_env_param: unknown field " + std::to_string(field));
  const std::string name = std::string("fb_set_env_param(") + kEnvParamName[field] + ")";
  if (!values) {                                    /* back to the model's value */
    if (h->ep_dev[field]) { dev_sync(h->stream); dev_free(h->ep_dev[field]); h->ep_dev[field] = nullptr; }
    h->ep_host[field].clear();
    env_param_bind(h);
    return field == FB_ENV_ACT_BIAS ? env_act_derive(h) : 0;
  }
  if ((field == FB_ENV_DRAG_COEF || field == FB_ENV_WATER_VELOCITY) && (!h->has_farms || h->ff_shallow.n_swim <= 0))
    return fail(name + ": the model has no swimming links");
  if (field == FB_ENV_CAND_FRICTION && h->fm_shallow.ncand <= 0) return fail(name + ": the model has no collision candidates");
  if ((field == FB_ENV_ACT_GAIN || field == FB_ENV_ACT_BIAS) && h->fm_shallow.nu <= 0) return fail(name + ": the model has no actuators");
  const FbModel &fm = h->fm_shallow;
  const int n = h->P.n_envs, w = env_param_width(h, field);
  const long long pad = h->P.env_pad;
  for (int e = 0; e < n; e++)
    for (int c = 0; c < w; c++) {
      const double v = values[(size_t)e*w + c];
      std::string at = " at environment " + std::to_string(e);
      if (field == FB_ENV_CAND_FRICTION) at += ", candidate " + std::to_string(c);
      else if (field == FB_ENV_ACT_GAIN) at += ", actuator " + std::to_string(c);
      else if (field == FB_ENV_ACT_BIAS) at += ", actuator " + std::to_string(c/3) + ", column " + std::to_string(c%3);
      else at += ", index " + std::to_string(c);
      /* drag coefficients are negative in FARMS (the force opposes the motion), a water velocity is
       * a vector, and MuJoCo checks no sign of a gain or bias (a <position kp> has bias -kp): only
       * stiffness and damping have a sign to check */
      const int signed_field = field == FB_ENV_DRAG_COEF || field == FB_ENV_WATER_VELOCITY ||
                               field == FB_ENV_ACT_GAIN || field == FB_ENV_ACT_BIAS;
      if (!std::isfinite(v)) return fail(name + ": non-finite value" + at);
      if (!signed_field && v < 0.0) return fail(name + ": negative value" + at);
      const int free_entry = (field == FB_ENV_JNT_STIFFNESS && fm.jnt_type[c] == FB_JNT_FREE) ||
                             (field == FB_ENV_DOF_DAMPING && fm.jnt_type[fm.dof_jntid[c]] == FB_JNT_FREE);
      if (free_entry && v != 0.0) return fail(name + ": non-zero value on the free joint" + at);
      if (field == FB_ENV_CAND_FRICTION) {
        /* an explicit <pair> takes its friction from the pair element, not from the geoms */
        const int pair = fm.cand_end[c] == 20 || fm.cand_end[c] == 21;
        if (pair && v != fm.cand_friction[c])
          return fail(name + ": " + std::to_string(v) + " differs from the <pair> candidate's friction " +
                      std::to_string(fm.cand_friction[c]) + at + " (pair frictions stay per model)");
        if (!pair && v < FB_MIN_ENV_FRICTION)
          return fail(name + ": friction " + std::to_string(v) + " below 0.1" + at + ": the pyramid rows stiffen as "
                      "1/mu^2 and the fp32 solver's error grows with them (3e-4 at mu = 0.1, 2.6e-3 at 0.05, "
                      "measured for pairs)");
      }
    }
  std::vector<float> dev((size_t)w*pad, 0.f);
  for (int e = 0; e < n; e++)
    for (int c = 0; c < w; c++) dev[(size_t)c*pad + e] = (float)values[(size_t)e*w + c];
  if (!h->ep_dev[field]) {
    void *p = nullptr;
    if (dev_alloc(&p, dev.size()*sizeof(float))) return fail(name + ": device allocation failed");
    h->ep_dev[field] = static_cast<float *>(p);
  }
  if (h2d(h->ep_dev[field], dev.data(), dev.size()*sizeof(float), h->stream) || dev_sync(h->stream))
    return fail(name + ": upload failed: " + dev_error());
  h->ep_host[field].assign(values, values + (size_t)n*w);
  env_param_bind(h);
  return field == FB_ENV_ACT_BIAS ? env_act_derive(h) : 0;
}

int fb_get_env_param(FbHandle *h, int field, double *out) {
  if (!h || !out) return fail("null argument");
  if (field < 0 || field >= FB_N_ENV_PARAM) return fail("fb_get_env_param: unknown field " + std::to_string(field));
  const int n = h->P.n_envs, w = env_param_width(h, field);
  if (h->ep_dev[field]) {
    std::copy(h->ep_host[field].begin(), h->ep_host[field].end(), out);
    return 0;
  }
  for (int e = 0; e < n; e++)
    for (int c = 0; c < w; c++) out[(size_t)e*w + c] = env_param_model(h, field, c);
  return 0;
}

int fb_set_swimming(FbHandle *h, int drag, int buoyancy) {
  if (!h) return fail("null handle");
  if (!h->has_farms) return fail("no farms tables");
  h->ff_shallow.water_drag = drag; h->ff_shallow.water_buoyancy = buoyancy;
  h->P.m.water_drag = h->hm.m.water_drag = drag != 0;
  h->P.m.water_buoyancy = h->hm.m.water_buoyancy = buoyancy != 0;
  return 0;
}

int fb_step(FbHandle *h, int n_steps, int want_derived, int sync) {
  if (!h) return fail("null handle");
  if (n_steps < 1) return fail("fb_step: n_steps must be >= 1");
  if (launch(h, FB_MODE_STEP, n_steps, want_derived)) return -1;
  if (sync && dev_sync(h->stream)) return fail(std::string("fb_step: ") + dev_error());
  return 0;
}

int fb_synchronize(FbHandle *h) {
  if (!h) return fail("null handle");
  return dev_sync(h->stream) ? fail(std::string("fb_synchronize: ") + dev_error()) : 0;
}

int fb_last_step_ms(FbHandle *h, float *ms) {
  if (!h || !ms) return fail("null argument");
#ifndef FB_HOST_EMU
  if (cudaEventSynchronize(h->ev1) != cudaSuccess) return fail(dev_error());
  if (cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1) != cudaSuccess) return fail(dev_error());
#endif
  *ms = h->last_ms;
  return 0;
}

int64_t fb_launch_count(FbHandle *h) { return h ? h->launches : 0; }

int fb_log_view(FbHandle *h, FbLogView *out) {
  if (!h || !out) return fail("null argument");
  const FbParams &P = h->P;
  out->links_dev = P.log_links; out->joints_dev = P.log_joints;
  out->contacts_dev = P.log_contacts; out->xfrc_dev = P.log_xfrc;
  out->links_vec = FB_VEC_LINKS; out->joints_vec = FB_VEC_JOINTS;
  out->contacts_vec = FB_VEC_CONTACTS; out->xfrc_vec = FB_VEC_XFRC;
  out->env_pad = (int32_t)P.env_pad;
  out->ring = P.ring; out->n_envs = P.n_envs;
  return 0;
}

int fb_state_view(FbHandle *h, FbStateView *out) {
  if (!h || !out) return fail("null argument");
  const FbParams &P = h->P;
  out->qpos_dev = P.qpos; out->qvel_dev = P.qvel; out->ctrl_dev = P.ctrl;
  out->xfrc_applied_dev = P.xfrc_applied; out->qpos_spring_dev = P.qpos_spring;
  out->env_phase_dev = P.env_phase; out->flags_dev = P.flags;
  out->iteration_dev = reinterpret_cast<int64_t *>(P.iteration);
  return 0;
}

int fb_derived_view(FbHandle *h, FbDerivedView *out) {
  if (!h || !out) return fail("null argument");
  const FbParams &P = h->P;
  out->xpos_dev = P.d_xpos; out->xquat_dev = P.d_xquat; out->xipos_dev = P.d_xipos;
  out->linvel_dev = P.d_linvel; out->angvel_dev = P.d_angvel; out->actuator_force_dev = P.d_actf;
  out->jnt_limit_force_dev = P.d_limf; out->qacc_dev = P.d_qacc; out->ncon_dev = P.d_ncon;
  out->con_cand_dev = P.d_con_cand; out->con_dist_dev = P.d_con_dist; out->con_pos_dev = P.d_con_pos;
  out->con_frame_dev = P.d_con_frame; out->con_force_dev = P.d_con_force;
  out->maxcon = h->hm.m.maxcon > 0 ? h->hm.m.maxcon : 1;
  return 0;
}

/* raw copies between host and the engine's device buffers (ctypes hosts
 * without torch use these; `what` selects the buffer) */
int fb_copy_to_host(FbHandle *h, const void *dev_ptr, void *host_ptr, int64_t bytes) {
  if (!h || !dev_ptr || !host_ptr) return fail("null argument");
  if (d2h(host_ptr, dev_ptr, (size_t)bytes, h->stream) || dev_sync(h->stream)) return fail(dev_error());
  return 0;
}
int fb_copy_to_device(FbHandle *h, void *dev_ptr, const void *host_ptr, int64_t bytes) {
  if (!h || !dev_ptr || !host_ptr) return fail("null argument");
  if (h2d(dev_ptr, host_ptr, (size_t)bytes, h->stream) || dev_sync(h->stream)) return fail(dev_error());
  return 0;
}

int fb_export_farms(FbHandle *h, int env, double *links, double *joints, double *contacts,
                    double *xfrc) {
  if (!h) return fail("null handle");
  const FbParams &P = h->P;
  if (env < 0 || env >= P.n_envs) return fail("fb_export_farms: env out of range");
  const DevModel &dm = h->hm.m;
  /* the environment's current episode: exported row r is ring row (s + r) % ring; when s > 0, rows
   * the episode has not reached (r > it - s) are zero */
  long long s = 0;
  if (d2h(&s, h->episode_start + env, sizeof(s), h->stream) || dev_sync(h->stream))
    return fail(std::string("fb_export_farms: ") + dev_error());
  const long long reached = h->it - s;
  struct Item { double *dst; const float *src; int row_floats, vec; } items[4] = {
    {links, P.log_links, dm.n_links*20, FB_VEC_LINKS},
    {joints, P.log_joints, dm.n_joints*dm.joint_cols, FB_VEC_JOINTS},
    {contacts, P.log_contacts, dm.n_contacts*12, FB_VEC_CONTACTS},
    {xfrc, P.log_xfrc, dm.n_xfrc*6, FB_VEC_XFRC}};
  for (const Item &it : items) {
    if (!it.dst || it.row_floats == 0) continue;
    const size_t count = (size_t)P.ring*it.row_floats;
    std::vector<float> tmp(count);
#ifdef FB_HOST_EMU
    for (size_t i = 0; i < count; i++) {
      size_t lin = i/it.vec;
      tmp[i] = it.src[(lin*P.env_pad + env)*it.vec + (i - lin*it.vec)];
    }
#else
    fb_gather_env_kernel<<<(unsigned)((count + 255)/256), 256, 0, h->stream>>>(
        it.src, P.ring, it.row_floats, it.vec, P.env_pad, env, h->gather_env);
    h->launches++;
    if (d2h(tmp.data(), h->gather_env, count*sizeof(float), h->stream) || dev_sync(h->stream))
      return fail(std::string("fb_export_farms: ") + dev_error());
#endif
    for (long long r = 0; r < P.ring; r++) {
      double *dst = it.dst + (size_t)r*it.row_floats;
      const float *src = tmp.data() + (size_t)((s + r) % P.ring)*it.row_floats;
      for (int i = 0; i < it.row_floats; i++) dst[i] = s > 0 && r > reached ? 0.0 : (double)src[i];
    }
  }
  return 0;
}

#ifndef FB_HOST_EMU
/* FARMS_B200_TRACE=1: device timeline of the pipelined host step (timing events on the three
 * streams of each call, printed by fb_host_wait); a debugging aid, off by default */
struct FbTraceCall { cudaEvent_t e[6]; double host_ms; };
static std::vector<FbTraceCall> g_trace;
static cudaEvent_t g_trace_t0;
static int g_trace_on = -1;
static double host_now_ms() {
  timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec*1e3 + ts.tv_nsec*1e-6;
}
static void trace_mark(int slot, cudaStream_t st) {
  if (g_trace_on != 1) return;
  cudaEventCreate(&g_trace.back().e[slot]);
  cudaEventRecord(g_trace.back().e[slot], st);
}
#endif

/* Shared body of fb_step_host / fb_step_host_async.  Asynchronous form: ctrl comes in on the upload
 * stream (SM reads of pinned host memory), the step kernels run on the handle's stream, the row
 * gathers and the two device->host copies on the copy stream, so the upload of launch i+1 and
 * the transfer of launch i overlap the kernels of launch i+1. */
static int step_host_impl(FbHandle *h, const float *ctrl, const float *qpos, const float *qvel,
                          int n_steps, float *links_row, float *joints_row, bool wait) {
  if (!h) return fail("null handle");
  FbParams &P = h->P;
  const DevModel &m = h->hm.m;
  const size_t n = (size_t)P.n_envs;
#ifndef FB_HOST_EMU
  if (g_trace_on < 0) g_trace_on = getenv("FARMS_B200_TRACE") ? 1 : 0;
  if (g_trace_on == 1) {
    if (g_trace.empty()) { cudaEventCreate(&g_trace_t0); cudaEventRecord(g_trace_t0, h->stream); }
    g_trace.push_back(FbTraceCall());
    for (auto &e : g_trace.back().e) e = nullptr;
    g_trace.back().host_ms = host_now_ms();
    trace_mark(0, h->stream);
  }
  bool ctrl_done = false;
  if (ctrl && m.nu > 0) {
    /* pinned (registered) host memory: the SMs fetch it on the upload stream while the previous
     * launch is still running; the launch stream then takes it over with a device copy */
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, ctrl) == cudaSuccess && pa.type == cudaMemoryTypeHost && pa.devicePointer) {
      const long long nf = (long long)n*(h->ctrl_sel_n > 0 ? h->ctrl_sel_n : m.nu);
      if (!h->ctrl_stage && alloc_arr(h, &h->ctrl_stage, (size_t)n*m.nu)) return fail("out of device memory (ctrl staging)");
      const float *src = static_cast<const float *>(pa.devicePointer);
      const int v4 = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(h->ctrl_stage) |
                       reinterpret_cast<uintptr_t>(P.ctrl)) & 15) == 0;
      if (cudaStreamWaitEvent(h->up_stream, h->ev_stage_free, 0) != cudaSuccess) return fail(dev_error());
      fb_copy_kernel<<<h->sms*2, 256, 0, h->up_stream>>>(src, h->ctrl_stage, nf, v4);
      if (cudaEventRecord(h->ev_up, h->up_stream) != cudaSuccess ||
          cudaStreamWaitEvent(h->stream, h->ev_up, 0) != cudaSuccess) return fail(dev_error());
      if (h->ctrl_sel_n > 0) {
        FbColSel sel;
        sel.n = h->ctrl_sel_n; sel.n_sel_items = 0;
        for (int k = 0; k < 32; k++) sel.col[k] = k < sel.n ? h->ctrl_sel[k] : 0;
        fb_scatter_ctrl_kernel<<<(unsigned)((nf + 255)/256), 256, 0, h->stream>>>(h->ctrl_stage, P.n_envs, m.nu, sel, P.ctrl);
      } else
      fb_copy_kernel<<<h->sms*4, 256, 0, h->stream>>>(h->ctrl_stage, P.ctrl, nf, v4);
      if (cudaEventRecord(h->ev_stage_free, h->stream) != cudaSuccess) return fail(dev_error());
      h->launches += 2;
      ctrl_done = true;
    } else {
      cudaGetLastError();               /* pageable memory: cudaPointerGetAttributes may flag it */
    }
  }
  if (ctrl && m.nu > 0 && !ctrl_done) {
    if (h->ctrl_sel_n > 0) {
      /* pageable memory: plain copy into the staging buffer, then the same scatter */
      const long long nf = (long long)n*h->ctrl_sel_n;
      if (!h->ctrl_stage && alloc_arr(h, &h->ctrl_stage, (size_t)n*m.nu)) return fail("out of device memory (ctrl staging)");
      if (h2d(h->ctrl_stage, ctrl, (size_t)nf*sizeof(float), h->stream)) return fail(dev_error());
      FbColSel sel;
      sel.n = h->ctrl_sel_n; sel.n_sel_items = 0;
      for (int k = 0; k < 32; k++) sel.col[k] = k < sel.n ? h->ctrl_sel[k] : 0;
      fb_scatter_ctrl_kernel<<<(unsigned)((nf + 255)/256), 256, 0, h->stream>>>(h->ctrl_stage, P.n_envs, m.nu, sel, P.ctrl);
      h->launches++;
    } else if (h2d(P.ctrl, ctrl, n*m.nu*sizeof(float), h->stream)) {
      return fail(dev_error());
    }
  }
#else
  if (ctrl && m.nu > 0) {
    if (h->ctrl_sel_n > 0) {
      for (size_t e = 0; e < n; e++)
        for (int k = 0; k < h->ctrl_sel_n; k++) P.ctrl[e*m.nu + h->ctrl_sel[k]] = ctrl[e*h->ctrl_sel_n + k];
    } else if (h2d(P.ctrl, ctrl, n*m.nu*sizeof(float), h->stream)) {
      return fail(dev_error());
    }
  }
#endif
  if (qpos && h2d(P.qpos, qpos, n*m.nq*sizeof(float), h->stream)) return fail(dev_error());
  if (qvel && h2d(P.qvel, qvel, n*m.nv*sizeof(float), h->stream)) return fail(dev_error());
#ifndef FB_HOST_EMU
  trace_mark(1, h->stream);
#endif
  if (launch(h, FB_MODE_STEP, n_steps, 0)) return -1;
#ifndef FB_HOST_EMU
  trace_mark(2, h->stream);
#endif
  long long row = h->it % P.ring;
  const bool link_sel = h->link_sel_n > 0 || h->link_items_n > 0;
  const int lsel_n = h->link_sel_n > 0 ? h->link_sel_n : 20, litems_n = h->link_items_n > 0 ? h->link_items_n : m.n_links;
  const int lf = litems_n*lsel_n;
  const int jf = m.n_joints*(h->joint_sel_n > 0 ? h->joint_sel_n : m.joint_cols);
#ifdef FB_HOST_EMU
  (void)wait;
  for (size_t e = 0; e < n; e++) {
    const int lsel = lsel_n, lfull = m.n_links*20;
    (void)link_sel;
    for (int i = 0; links_row && i < lf; i++) {
      const int oi = i/lsel, c = h->link_sel_n > 0 ? h->link_sel[i - oi*lsel] : i - oi*lsel;
      const int item = h->link_items_n > 0 ? h->link_items[oi] : oi;
      const long long f = (long long)item*20 + c, g = f/FB_VEC_LINKS;
      links_row[e*lf + i] = P.log_links[((row*(lfull/FB_VEC_LINKS) + g)*P.env_pad + e)*FB_VEC_LINKS + f % FB_VEC_LINKS];
    }
    const int nsel = h->joint_sel_n > 0 ? h->joint_sel_n : m.joint_cols, jfull = m.n_joints*m.joint_cols;
    for (int i = 0; joints_row && i < jf; i++) {
      const int item = i/nsel, c = h->joint_sel_n > 0 ? h->joint_sel[i - item*nsel] : i - item*nsel;
      const long long f = (long long)item*m.joint_cols + c, g = f/FB_VEC_JOINTS;
      joints_row[e*jf + i] = P.log_joints[((row*(jfull/FB_VEC_JOINTS) + g)*P.env_pad + e)*FB_VEC_JOINTS + f % FB_VEC_JOINTS];
    }
  }
#else
  const bool want_links = links_row && lf, want_joints = joints_row && jf;
  if (want_links || want_joints) {
    /* gathers on the gather stream behind this call's kernels, copies on the copy stream behind
     * the gathers: the launch stream goes straight on to the next call's kernels (launch() orders
     * them against these gathers), and two pairs of gather buffers let the gathers of this call
     * run while the copies of the previous one are still on the bus */
    const int slot = (int)(h->host_calls & 3), pair = (int)(h->host_calls & 1);
    if (pair && !h->gather_links2) {
      if (alloc_arr(h, &h->gather_links2, n*m.n_links*20) || alloc_arr(h, &h->gather_joints2, n*m.n_joints*m.joint_cols))
        return fail("out of device memory (second pair of gather buffers)");
    }
    float *g_links = pair ? h->gather_links2 : h->gather_links, *g_joints = pair ? h->gather_joints2 : h->gather_joints;
    cudaStream_t cs = h->gather_stream;
    /* this pair of gather buffers was last used two calls ago: its copies must have left */
    if (h->host_calls >= 2 && cudaStreamWaitEvent(cs, h->ev_copy[(slot + 2) & 3], 0) != cudaSuccess) return fail(dev_error());
    h->host_calls++;
    if (cudaEventRecord(h->ev_gather, h->stream) != cudaSuccess ||
        cudaStreamWaitEvent(cs, h->ev_gather, 0) != cudaSuccess) return fail(dev_error());
    trace_mark(4, cs);
    if (want_links && link_sel) {
      FbColSel sel;
      sel.n = lsel_n;
      for (int k = 0; k < 32; k++) sel.col[k] = h->link_sel_n > 0 ? (k < sel.n ? h->link_sel[k] : 0) : (k < 20 ? k : 0);
      sel.n_sel_items = h->link_items_n;
      for (int k = 0; k < 64; k++) sel.item[k] = k < h->link_items_n ? h->link_items[k] : 0;
      long long total = (long long)n*lf;
      fb_gather_cols_kernel<<<(unsigned)((total + 255)/256), 256, 0, cs>>>(
          P.log_links, row, m.n_links, 20, FB_VEC_LINKS, P.env_pad, P.n_envs, sel, g_links);
      h->launches++;
    } else if (want_links) {
      const int nvec = lf/FB_VEC_LINKS;
      static_assert(FB_VEC_LINKS == 4, "fb_gather_rows4_kernel moves float4 vectors");
      fb_gather_rows4_kernel<<<dim3((unsigned)((n + 31)/32), (unsigned)((nvec + 31)/32)), 256, 0, cs>>>(
          reinterpret_cast<const float4 *>(P.log_links), row, nvec, P.env_pad, P.n_envs,
          reinterpret_cast<float4 *>(g_links));
      h->launches++;
    }
    if (want_joints && h->joint_sel_n > 0) {
      FbColSel sel;
      sel.n = h->joint_sel_n;
      sel.n_sel_items = 0;
      for (int k = 0; k < 32; k++) sel.col[k] = k < sel.n ? h->joint_sel[k] : 0;
      long long total = (long long)n*jf;
      fb_gather_cols_kernel<<<(unsigned)((total + 255)/256), 256, 0, cs>>>(
          P.log_joints, row, m.n_joints, m.joint_cols, FB_VEC_JOINTS, P.env_pad, P.n_envs, sel, g_joints);
      h->launches++;
    } else if (want_joints) {
      long long total = (long long)n*(jf/FB_VEC_JOINTS);
      fb_gather_rows_kernel<<<(unsigned)((total + 255)/256), 256, 0, cs>>>(
          P.log_joints, row, jf, FB_VEC_JOINTS, P.env_pad, P.n_envs, g_joints);
      h->launches++;
    }
    if (cudaEventRecord(h->ev_gathered[slot], cs) != cudaSuccess) return fail(dev_error());
    h->gather_it[slot] = h->it;
    trace_mark(3, cs);
    cs = h->copy_stream;
    if (cudaStreamWaitEvent(cs, h->ev_gathered[slot], 0) != cudaSuccess) return fail(dev_error());
    if (want_links && d2h(links_row, g_links, (size_t)n*lf*sizeof(float), cs)) return fail(dev_error());
    if (want_joints && d2h(joints_row, g_joints, (size_t)n*jf*sizeof(float), cs)) return fail(dev_error());
    if (cudaEventRecord(h->ev_copy[slot], cs) != cudaSuccess) return fail(dev_error());
    trace_mark(5, cs);
  }
  if (wait) {
    if (cudaStreamSynchronize(h->copy_stream) != cudaSuccess) return fail(dev_error());
  }
#endif
  if (wait && dev_sync(h->stream)) return fail(std::string("fb_step_host: ") + dev_error());
  return 0;
}

int fb_step_host(FbHandle *h, const float *ctrl, const float *qpos, const float *qvel,
                 int n_steps, float *links_row, float *joints_row) {
  return step_host_impl(h, ctrl, qpos, qvel, n_steps, links_row, joints_row, true);
}

int fb_step_host_async(FbHandle *h, const float *ctrl, const float *qpos, const float *qvel,
                       int n_steps, float *links_row, float *joints_row) {
  return step_host_impl(h, ctrl, qpos, qvel, n_steps, links_row, joints_row, false);
}

/* Wait for the copies of the latest pipelined call with (call index % 2) == slot. */
int fb_host_wait_slot(FbHandle *h, int slot) {
  if (!h) return fail("null handle");
#ifndef FB_HOST_EMU
  long long call = h->host_calls - 1;
  if ((call & 1) != (slot & 1)) call--;
  if (call >= 0 && cudaEventSynchronize(h->ev_copy[call & 3]) != cudaSuccess) return fail(dev_error());
#else
  (void)slot;
#endif
  return 0;
}

/* Calls of fb_step_host / fb_step_host_async that asked for rows so far: the next one has this index. */
long long fb_host_call_count(FbHandle *h) {
#ifndef FB_HOST_EMU
  return h ? h->host_calls : 0;
#else
  (void)h; return 0;
#endif
}

/* Wait for the copies of pipelined call `call` (index as counted by fb_host_call_count).  The
 * copies complete in call order, so an index older than the four-event ring waits on a later
 * call's event, which implies its own. */
int fb_host_wait_call(FbHandle *h, long long call) {
  if (!h) return fail("null handle");
#ifndef FB_HOST_EMU
  if (call >= h->host_calls) return fail("fb_host_wait_call: no such call yet");
  if (call >= 0 && cudaEventSynchronize(h->ev_copy[call & 3]) != cudaSuccess) return fail(dev_error());
#else
  (void)call;
#endif
  return 0;
}

int fb_host_wait(FbHandle *h) {
  if (!h) return fail("null handle");
#ifndef FB_HOST_EMU
  if (cudaStreamSynchronize(h->copy_stream) != cudaSuccess) return fail(dev_error());
  if (g_trace_on == 1 && !g_trace.empty()) {
    cudaStreamSynchronize(h->stream);
    const double h0 = g_trace[0].host_ms;
    fprintf(stderr, "call  host_enq | main: begin  ctrl_in  kernels | copy: gathered | start  done   (ms)\n");
    for (size_t c = 0; c < g_trace.size(); c++) {
      fprintf(stderr, "%4zu  %8.3f |", c, g_trace[c].host_ms - h0);
      for (int k = 0; k < 6; k++) {
        float ms = -1.f;
        if (g_trace[c].e[k]) { cudaEventElapsedTime(&ms, g_trace_t0, g_trace[c].e[k]); cudaEventDestroy(g_trace[c].e[k]); }
        fprintf(stderr, " %8.3f%s", ms, k == 3 ? " |" : "");
      }
      fprintf(stderr, "\n");
    }
    cudaEventDestroy(g_trace_t0);
    g_trace.clear();
  }
#endif
  return dev_sync(h->stream) ? fail(std::string("fb_host_wait: ") + dev_error()) : 0;
}

int fb_set_host_joint_columns(FbHandle *h, int n, const int32_t *cols) {
  if (!h) return fail("null handle");
  if (n < 0 || n > 32 || (n > 0 && !cols)) return fail("fb_set_host_joint_columns: 0..32 columns");
  for (int k = 0; k < n; k++)
    if (cols[k] < 0 || cols[k] >= h->hm.m.joint_cols) return fail("fb_set_host_joint_columns: column out of range");
  /* the pipelined copies of earlier calls used the previous row width */
  if (fb_host_wait(h)) return -1;
  h->joint_sel_n = n;
  for (int k = 0; k < n; k++) h->joint_sel[k] = cols[k];
  return 0;
}

int fb_set_host_link_columns(FbHandle *h, int n, const int32_t *cols) {
  if (!h) return fail("null handle");
  if (n < 0 || n > 20 || (n > 0 && !cols)) return fail("fb_set_host_link_columns: 0..20 columns");
  for (int k = 0; k < n; k++)
    if (cols[k] < 0 || cols[k] >= 20) return fail("fb_set_host_link_columns: column out of range");
  if (fb_host_wait(h)) return -1;
  h->link_sel_n = n;
  for (int k = 0; k < n; k++) h->link_sel[k] = cols[k];
  return 0;
}

int fb_set_host_ctrl_columns(FbHandle *h, int n, const int32_t *cols) {
  if (!h) return fail("null handle");
  if (n < 0 || n > 32 || (n > 0 && !cols)) return fail("fb_set_host_ctrl_columns: 0..32 actuators");
  for (int k = 0; k < n; k++)
    if (cols[k] < 0 || cols[k] >= h->hm.m.nu) return fail("fb_set_host_ctrl_columns: actuator out of range");
  if (fb_host_wait(h)) return -1;
  h->ctrl_sel_n = n;
  for (int k = 0; k < n; k++) h->ctrl_sel[k] = cols[k];
  return 0;
}

int fb_set_host_link_items(FbHandle *h, int n, const int32_t *items) {
  if (!h) return fail("null handle");
  if (n < 0 || n > 64 || (n > 0 && !items)) return fail("fb_set_host_link_items: 0..64 links");
  for (int k = 0; k < n; k++)
    if (items[k] < 0 || items[k] >= h->hm.m.n_links) return fail("fb_set_host_link_items: link out of range");
  if (fb_host_wait(h)) return -1;
  h->link_items_n = n;
  for (int k = 0; k < n; k++) h->link_items[k] = items[k];
  return 0;
}

/* Streamed export of whole ring rows: rows row0 .. row0+n_rows-1 (ring indices, modulo the ring)
 * of one log kind for EVERY environment, as dense float32 [n_rows][n_envs][n_items*n_cols] on the
 * host -- per environment and row exactly data.sensors.<kind>.array[row] (task.py:158).  Each row
 * is transposed out of the environment-minor log by a gather kernel into one of two staging
 * buffers and copied down on the copy stream while the next row is gathered. */
int fb_export_rows(FbHandle *h, int kind, int row0, int n_rows, float *host) {
  if (!h || !host) return fail("null argument");
  const FbParams &P = h->P;
  const DevModel &m = h->hm.m;
  if (kind < 0 || kind > 3) return fail("fb_export_rows: kind 0 links, 1 joints, 2 contacts, 3 xfrc");
  if (n_rows < 1 || n_rows > P.ring || row0 < 0) return fail("fb_export_rows: bad row range");
  const float *src[4] = {P.log_links, P.log_joints, P.log_contacts, P.log_xfrc};
  const int floats[4] = {m.n_links*20, m.n_joints*m.joint_cols, m.n_contacts*12, m.n_xfrc*6};
  const int vec[4] = {FB_VEC_LINKS, FB_VEC_JOINTS, FB_VEC_CONTACTS, FB_VEC_XFRC};
  const int rf = floats[kind];
  if (rf == 0) return 0;
  const size_t n = (size_t)P.n_envs, per_row = n*rf;
#ifdef FB_HOST_EMU
  for (int r = 0; r < n_rows; r++) {
    const long long row = (row0 + r) % P.ring;
    for (size_t e = 0; e < n; e++)
      for (int i = 0; i < rf; i++) {
        const long long g = i/vec[kind];
        host[(size_t)r*per_row + e*rf + i] = src[kind][((row*(rf/vec[kind]) + g)*P.env_pad + e)*vec[kind] + i % vec[kind]];
      }
  }
  return 0;
#else
  if (dev_sync(h->stream)) return fail(dev_error());       /* the rows are complete */
  if (h->export_stage_floats < per_row) {
    for (int k = 0; k < 2; k++) {
      if (h->export_stage[k]) cudaFree(h->export_stage[k]);
      if (cudaMalloc(&h->export_stage[k], per_row*sizeof(float)) != cudaSuccess) {
        h->export_stage[k] = nullptr; h->export_stage_floats = 0;
        return fail("fb_export_rows: out of device memory (staging)");
      }
    }
    h->export_stage_floats = per_row;
  }
  cudaEvent_t gathered[2], copied[2];
  for (int k = 0; k < 2; k++) {
    cudaEventCreateWithFlags(&gathered[k], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&copied[k], cudaEventDisableTiming);
  }
  int rc = 0;
  for (int r = 0; r < n_rows && !rc; r++) {
    const int b = r & 1;
    const long long row = (row0 + r) % P.ring;
    if (r >= 2) cudaStreamWaitEvent(h->gather_stream, copied[b], 0);   /* the staging buffer is free again */
    if (vec[kind] == 4) {
      const int nvec = rf/4;
      fb_gather_rows4_kernel<<<dim3((unsigned)((n + 31)/32), (unsigned)((nvec + 31)/32)), 256, 0, h->gather_stream>>>(
          reinterpret_cast<const float4 *>(src[kind]), row, nvec, P.env_pad, P.n_envs,
          reinterpret_cast<float4 *>(h->export_stage[b]));
    } else {
      const long long total = (long long)n*(rf/vec[kind]);
      fb_gather_rows_kernel<<<(unsigned)((total + 255)/256), 256, 0, h->gather_stream>>>(
          src[kind], row, rf, vec[kind], P.env_pad, P.n_envs, h->export_stage[b]);
    }
    h->launches++;
    cudaEventRecord(gathered[b], h->gather_stream);
    cudaStreamWaitEvent(h->copy_stream, gathered[b], 0);
    if (d2h(host + (size_t)r*per_row, h->export_stage[b], per_row*sizeof(float), h->copy_stream)) rc = -1;
    cudaEventRecord(copied[b], h->copy_stream);
  }
  if (cudaStreamSynchronize(h->copy_stream) != cudaSuccess || cudaGetLastError() != cudaSuccess) rc = -1;
  for (int k = 0; k < 2; k++) { cudaEventDestroy(gathered[k]); cudaEventDestroy(copied[k]); }
  return rc ? fail(std::string("fb_export_rows: ") + dev_error()) : 0;
#endif
}

int fb_set_fast_path(FbHandle *h, int enable) {
  if (!h) return fail("null handle");
  h->fast_enabled = enable != 0;
  return 0;
}
int fb_set_constraint_path(FbHandle *h, int per_thread) {
  if (!h) return fail("null handle");
  h->con_thread = per_thread != 0;
  return 0;
}
int fb_constraint_path(FbHandle *h) { return h && fb_next_step(h).con_thread ? 1 : 0; }
/* 0: team kernel only; otherwise the environments per block of the per-thread kernel */
int fb_fast_path(FbHandle *h) {
  if (!h) return 0;
  const FbPlan p = fb_next_step(h);
  return p.fast ? p.uncon.blk : 0;
}
int fb_fast_smem_bytes_per_env(FbHandle *h) {
  return h ? (int)((h->fast_slim ? h->hm.m.X.n_float_slim : h->hm.m.X.n_float)*sizeof(float)) : 0;
}
/* 0: regular layout; else the warps per block of the large-batch (SLIM) layout (1 .. 8) */
int fb_fast_slim(FbHandle *h) {
  if (!h) return 0;
  const FbPlan p = fb_next_step(h);
  return p.fast && p.uncon.slim ? p.uncon.threads/32 : 0;
}
int fb_set_fast_slim(FbHandle *h, int enable) {
  if (!h) return fail("null handle");
  if (enable < 0 || enable > 8) return fail("fb_set_fast_slim: 0 (regular layout) or 1 .. 8 warps per block");
  h->fast_wpb = enable > 1 ? enable : 1;
#ifndef FB_HOST_EMU
  if (enable && h->fast_block != 32) return fail("fb_set_fast_slim: needs 32 environments per warp");
  if (enable && fb_slim_attributes(h)) return -1;
#endif
  h->fast_slim = enable != 0;
  return 0;
}
/* SPLIT variant of the unconstrained kernel (small batches): several warps per 32 environments */
int fb_set_fast_split(FbHandle *h, int enable) {
  if (!h) return fail("null handle");
  h->fast_split = enable != 0;
  return 0;
}
/* warps per 32 environments when fb_step launches the SPLIT variant, else 0 (the batch must fit one
 * wave of its blocks; while fb_create's 16-per-warp guess stands -- until the first launch of an
 * episode has been reviewed -- the single-warp kernels run) */
int fb_fast_split(FbHandle *h) {
  if (!h) return 0;
  const FbPlan p = fb_next_step(h);
  return p.fast && p.uncon.kind == FB_FAST_SPLIT ? h->hm.split.nwarps : 0;
}
/* drag_forces (swimming/drag.pyx:152-268) as a stand-alone device operator, see include/farms_b200.h */
int fb_drag_forces(int device, int n, const double *links, const double *coefficients, const double *mass,
                   const double *height, const double *density, double surface, const double *water_velocity,
                   double viscosity, double gravity, int use_buoyancy, double *xfrc, int32_t *applied) {
  if (n < 0 || (n > 0 && (!links || !coefficients || !mass || !height || !density || !water_velocity || !xfrc || !applied)))
    return fail("fb_drag_forces: null argument");
  if (n == 0) return 0;
  FbDragArgs A;
  A.surface = surface; A.viscosity = viscosity; A.gravity = gravity;
  for (int k = 0; k < 3; k++) A.wvel[k] = water_velocity[k];
  A.use_buoyancy = use_buoyancy != 0; A.n = n;
#ifdef FB_HOST_EMU
  (void)device;
  std::vector<int> flags((size_t)n);
  A.links = links; A.coef = coefficients; A.mass = mass; A.height = height; A.density = density;
  A.xfrc = xfrc; A.applied = flags.data();
  for (int i = 0; i < n; i++) { fb_drag_row(A, i); applied[i] = flags[(size_t)i]; }
  return 0;
#else
  if (cudaSetDevice(device) != cudaSuccess) return fail(std::string("fb_drag_forces: ") + dev_error());
  const size_t nn = (size_t)n;
  const size_t bytes_in = nn*(20 + 6 + 3)*sizeof(double), bytes_out = nn*6*sizeof(double) + nn*sizeof(int);
  void *din = nullptr, *dout = nullptr;
  if (dev_alloc(&din, bytes_in) || dev_alloc(&dout, bytes_out)) { if (din) dev_free(din); return fail("fb_drag_forces: device allocation failed"); }
  double *d_links = static_cast<double *>(din), *d_coef = d_links + 20*nn, *d_mass = d_coef + 6*nn,
         *d_height = d_mass + nn, *d_density = d_height + nn;
  double *d_xfrc = static_cast<double *>(dout);
  int *d_applied = reinterpret_cast<int *>(d_xfrc + 6*nn);
  cudaError_t ce = cudaMemcpy(d_links, links, 20*nn*sizeof(double), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMemcpy(d_coef, coefficients, 6*nn*sizeof(double), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMemcpy(d_mass, mass, nn*sizeof(double), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMemcpy(d_height, height, nn*sizeof(double), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMemcpy(d_density, density, nn*sizeof(double), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMemcpy(d_xfrc, xfrc, 6*nn*sizeof(double), cudaMemcpyHostToDevice);     /* rows that are not applied keep their values */
  if (ce == cudaSuccess) {
    A.links = d_links; A.coef = d_coef; A.mass = d_mass; A.height = d_height; A.density = d_density;
    A.xfrc = d_xfrc; A.applied = d_applied;
    fb_drag_forces_kernel<<<(n + 127)/128, 128>>>(A);
    ce = cudaGetLastError();
  }
  if (ce == cudaSuccess) ce = cudaMemcpy(xfrc, d_xfrc, 6*nn*sizeof(double), cudaMemcpyDeviceToHost);
  if (ce == cudaSuccess) ce = cudaMemcpy(applied, d_applied, nn*sizeof(int), cudaMemcpyDeviceToHost);
  dev_free(din); dev_free(dout);
  return ce == cudaSuccess ? 0 : fail(std::string("fb_drag_forces: ") + cudaGetErrorString(ce));
#endif
}

/* SPLIT variant of the constrained per-thread kernel (ground-contact batches) */
int fb_set_con_split(FbHandle *h, int enable) {
  if (!h) return fail("fb_set_con_split: null handle");
  h->con_split = enable != 0;
  return 0;
}

/* 1 when the next launch hands the fully handed-over groups to the SPLIT variant */
int fb_con_split(FbHandle *h) { return h && fb_next_step(h).con_split ? 1 : 0; }

/* resident SPLIT blocks per SM as the runtime computes it (0: not applicable) */
int fb_fast_split_blocks_per_sm(FbHandle *h) {
#ifndef FB_HOST_EMU
  if (!h || !h->hm.m.X.ok || h->hm.split.nwarps < 2) return 0;
  int nb = 0;
  return fb_kernel_attributes(fb_kernel_sel(h, FB_FAST_SPLIT, 32), &nb) == cudaSuccess ? nb : 0;
#else
  (void)h; return 0;
#endif
}
/* the schedule itself (tests): n[4], boundary[4], order[4][64]; returns the number of warps */
int fb_fast_split_schedule(FbHandle *h, int32_t *n, int32_t *boundary, uint8_t *order) {
  if (!h || !n || !boundary || !order) return 0;
  const FastSplit &sp = h->hm.split;
  for (int w = 0; w < FB_SPLIT_MAXW; w++) { n[w] = sp.n[w]; boundary[w] = sp.boundary[w]; }
  memcpy(order, sp.order, sizeof(sp.order));
  return sp.nwarps;
}
/* LEAN variants of the unconstrained kernel (fb_fast.h): on by default when the model allows */
int fb_set_fast_lean(FbHandle *h, int enable) {
  if (!h) return fail("null handle");
  h->fast_lean = enable != 0;
  return 0;
}
/* 1 when fb_step launches the LEAN variant for this model (a control sequence falls back) */
int fb_fast_lean(FbHandle *h) {
  if (!h) return 0;
  const FbPlan p = fb_next_step(h);
  return p.fast && p.uncon.lean ? 1 : 0;
}
/* environments the team kernel had to finish in the last fb_step (synchronises) */
int fb_last_pending(FbHandle *h, int *count) {
  if (!h || !count) return fail("null argument");
  int both[2] = {0, 0};
  if (d2h(both, h->P.pending_count, sizeof(both), h->stream) || dev_sync(h->stream)) return fail(dev_error());
  *count = h->P.use_pending ? both[h->P.parity] : h->P.n_envs;
  return 0;
}

#ifdef FB_HOST_EMU
/* emulation harness only: counters of the per-thread constrained solver */
void fb_emu_solver_stats(double *stats3) { fb_emu_stats = stats3; }
#endif

/* measured FFMA throughput of `device` in TFLOP/s (2 flops per FFMA), best of 5 launches */
int fb_measure_fp32_peak(int device, double *tflops_out) {
  if (!tflops_out) return fail("null argument");
#ifdef FB_HOST_EMU
  (void)device; *tflops_out = 0.0;
  return fail("fb_measure_fp32_peak: needs a CUDA device");
#else
  int sms = 0;
  if (cudaSetDevice(device) != cudaSuccess ||
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return fail(dev_error());
  float *out = nullptr;
  cudaEvent_t e0, e1;
  if (cudaMalloc(&out, sizeof(float)) != cudaSuccess) return fail(dev_error());
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  const int blocks = sms*8, iters = 2048;         /* 8 x 256 threads = 64 warps per SM in flight */
  double best = 0.0;
  for (int rep = 0; rep < 6; rep++) {
    cudaEventRecord(e0, 0);
    fb_ffma_peak_kernel<<<blocks, 256>>>(out, iters, 1.0f, 1e-9f);
    cudaEventRecord(e1, 0);
    if (cudaEventSynchronize(e1) != cudaSuccess) { cudaFree(out); return fail(dev_error()); }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double tf = 2.0*8*16*(double)iters*256.0*blocks/(ms*1e-3)*1e-12;
    if (rep && tf > best) best = tf;              /* first launch: warm-up */
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
  *tflops_out = best;
  return 0;
#endif
}

int fb_team_lanes(FbHandle *h) { return h ? h->team : 0; }
int fb_smem_bytes_per_env(FbHandle *h) {
  return h ? (int)((h->hm.m.L.n_float + h->hm.m.L.n_int)*sizeof(float)) : 0;
}
int fb_device_ptr_stream(FbHandle *h, void **stream_out) {
  if (!h || !stream_out) return fail("null argument");
#ifdef FB_HOST_EMU
  *stream_out = nullptr;
#else
  *stream_out = (void *)h->stream;
#endif
  return 0;
}

}  /* extern "C" */
