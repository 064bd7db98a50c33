// libgrasp_engine.so — C-ABI (include/grasp_engine.h) + kernels of the batched grasp-simulation engine.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC (see __graft_entry__.build()).
#include "ge_variant.h"  // must come first: renames the namespace and the C entry points of this build variant

#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/grasp_engine.h"
#include "ge_render.cuh"
#include "ge_step.cuh"

using namespace ge;

static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, const char* a = "") { snprintf(g_err, sizeof g_err, fmt, a); return code; }
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(GE_ERR_CUDA, "CUDA error: %s", cudaGetErrorString(e_)); } while (0)

extern "C" const char* ge_last_error(void) { return g_err; }
extern "C" const char* ge_version(void) { return GE_NW > 1 ? "grasp_engine 0.3 sm_100a fp64 CTA-per-env (4 warps, workspace: shared memory, Hessian overflow: HBM)" : "grasp_engine 0.3 sm_100a fp64 warp-per-env (workspace: shared memory)"; }

// ------------------------------------------------------------------------------------------------ kernels
// Sub-step kernel: one warp per environment, environments handed to warps DYNAMICALLY.
// A launch gives every environment a budget of `nsub` iterations of the reference control loop (PID -> mj_step, including the
// movement / grasp-program transitions), split into visits of `quota` iterations.  Task t of a launch = (visit t / n_env, env t % n_env);
// a warp that has no environment takes the next task from a global counter, skips it if the environment is idle, hands its
// iterations to the warp that still runs an earlier visit of it (per-env lock word: bit 0 held, the rest handed-over iterations; the
// holder runs them before it lets go), otherwise loads the env's state rows into its shared-memory slice, runs the visit and writes
// the rows back.  No iteration of a busy env is dropped, so every env runs its whole budget (or until it goes idle) and what a launch
// computes does not depend on timing.  The grid is persistent (<= the resident CTAs), so 4096 envs on 1184 warp slots cost 13.84 -> 14
// rounds of 64 iterations instead of 3.46 -> 4 rounds of 256, finished or idle environments stop costing anything, and the tail
// of a batch of unequal grasp attempts is spread over all SMs.  Arithmetic per env is unchanged: the state crosses HBM in full
// fp64 between visits, so a trajectory does not depend on how its iterations were cut.
// A CTA holds `blockDim.y` warps; they meet at one barrier per iteration (+ the stage barriers) so that the warps of an SM walk
// the (large) sub-step code roughly together and share instruction-cache lines.
namespace ge {
struct EnvRegs {
  Cmd c; Prog p; int info[12]; unsigned char reward; int status; long long nstep;
};
__device__ __forceinline__ bool env_is_busy(const EnvArrays& E, int env) { return __ldcg(E.cmd_active + env) != 0 || __ldcg(E.prog_phase + env) != PH_NONE; }
__device__ __forceinline__ void env_load(const EnvArrays& E, int env, double* ws, int lane, EnvRegs& r) {
  const DevModel& m = c_m; const Layout& L = c_L;
  r.c.active = __ldcg(E.cmd_active + env); r.p.phase = __ldcg(E.prog_phase + env);
  r.c.mask = __ldcg(E.cmd_mask + env); r.c.maxsteps = __ldcg(E.cmd_maxsteps + env); r.c.steps = __ldcg(E.cmd_steps + env);
  r.c.result = __ldcg(E.cmd_result + env); r.c.tol = __ldcg(E.cmd_tol + env); r.c.reached = 0;
  int aux = __ldcg(E.prog_aux + env);
  r.p.rot = __ldcg(E.prog_rot + env); r.p.grasp = __ldcg(E.prog_grasp + env); r.p.aux = aux & 0xffff; r.p.r1 = (aux >> 16) & 0xf; r.p.rfinal = ((aux >> 20) & 0xf) - 1;
  for (int k = 0; k < 3; k++) r.p.coords[k] = __ldcg(E.prog_coords + 3 * env + k);
  r.p.table = __ldcg(E.prog_table + env);
  for (int k = 0; k < 12; k++) r.info[k] = __ldcg(E.prog_info + 12 * env + k);
  r.reward = __ldcg(E.reward + env); r.status = __ldcg(E.status + env); r.nstep = 0;
  LANE_LOOP(i, m.nq) ws[L.qpos + i] = __ldcg(E.qpos + (size_t)env * m.nq + i);
  LANE_LOOP(i, m.nv) { ws[L.qvel + i] = __ldcg(E.qvel + (size_t)env * m.nv + i); ws[L.qaccws + i] = __ldcg(E.qaccws + (size_t)env * m.nv + i); }
  if (lane < 32) ws[L.ctl + lane] = __ldcg(E.ctl + (size_t)env * 32 + lane);
  gsync();
}
__device__ __forceinline__ void env_store(const EnvArrays& E, int env, const double* ws, int lane, const EnvRegs& r) {
  const DevModel& m = c_m; const Layout& L = c_L;
  LANE_LOOP(i, m.nq) E.qpos[(size_t)env * m.nq + i] = ws[L.qpos + i];
  LANE_LOOP(i, m.nv) { E.qvel[(size_t)env * m.nv + i] = ws[L.qvel + i]; E.qaccws[(size_t)env * m.nv + i] = ws[L.qaccws + i]; }
  if (lane < 32) E.ctl[(size_t)env * 32 + lane] = ws[L.ctl + lane];
  if (lane == 0) {
    E.cmd_active[env] = r.c.active; E.cmd_mask[env] = r.c.mask; E.cmd_maxsteps[env] = r.c.maxsteps; E.cmd_steps[env] = r.c.steps;
    E.cmd_result[env] = r.c.result; E.cmd_tol[env] = r.c.tol;
    E.prog_phase[env] = r.p.phase; E.prog_grasp[env] = r.p.grasp;
    E.prog_aux[env] = (r.p.aux & 0xffff) | ((r.p.r1 & 0xf) << 16) | (((r.p.rfinal + 1) & 0xf) << 20);
    for (int k = 0; k < 12; k++) E.prog_info[12 * env + k] = r.info[k];
    E.reward[env] = r.reward; E.status[env] = r.status; E.substeps[env] += r.nstep;
  }
}

__device__ __forceinline__ unsigned long long group_bcast_u64(unsigned long long v, int lane) {
#if GE_NW == 1
  return __shfl_sync(FULL, v, 0);
#else
  __shared__ unsigned long long b;
  if (lane == 0) b = v;
  cta_sync();
  unsigned long long r = b;
  cta_sync();
  return r;
#endif
}
// blockDim = (GE_LANES, envs per CTA): threadIdx.x is the lane inside the group that owns one environment (a warp; a whole CTA of
// GE_NW warps in the big-scene build, where blockDim.y = 1)
// Register budget.  Warp-per-env build: `__launch_bounds__(256)` alone makes ptxas settle on 128 registers per thread (stack 1616 B); told
// that one 256-thread CTA per SM is enough it takes 246 (stack 1296 B), which still fits the 2 x 128-thread CTAs the shared memory allows
// (65 536 registers per SM) - r02g: 3.93 -> 4.20 M sub-steps/s at 4096 envs (-DGE_V0_CAP_REGS restores the old budget).
// CTA-per-env build: two CTAs per SM is what the workspace allows; the bound keeps the register file from undercutting it.
#if GE_NW > 1
#define GE_RUN_BOUNDS __launch_bounds__(GE_LANES, 2)
#elif defined(GE_V0_CAP_REGS)
#define GE_RUN_BOUNDS __launch_bounds__(256)
#else
#define GE_RUN_BOUNDS __launch_bounds__(256, 1)
#endif
__global__ void GE_RUN_BOUNDS k_run(EnvArrays E, int n_env, int nsub, int quota, unsigned long long ticket_base, double base_x, double base_y,
                                             double base_z, int stage_sync) {
  extern __shared__ double smem[];
  const Layout& L = c_L;
  const int lane = threadIdx.x;
  const int visits = (nsub + quota - 1) / quota;
  const unsigned long long total = (unsigned long long)n_env * visits;
  const double base[3] = {base_x, base_y, base_z};
  double* ws = smem + (size_t)threadIdx.y * (L.total_bytes / 8);
  int* wi = (int*)(ws + L.total_doubles);
  EnvRegs r;
  int env = -1, left = 0;
  bool exhausted = false, running = false;
  for (;;) {
    // ---- a group without an environment takes tasks until it finds a busy, unlocked environment (or the launch has none left)
    while (env < 0 && !exhausted) {
      unsigned long long t = 0;
      if (lane == 0) t = atomicAdd(E.ticket, 1ULL) - ticket_base;
      t = group_bcast_u64(t, lane);
      if (t >= total) { exhausted = true; break; }
      const int e = (int)(t % (unsigned long long)n_env), v = (int)(t / (unsigned long long)n_env);
      const int n_it = nsub - v * quota < quota ? nsub - v * quota : quota;
      // ONE thread takes the lock and looks at the env's flags, the group follows its verdict: the flags change under our feet when
      // another group finishes a visit of this env, and threads that read them separately (the four warps of a CTA-per-env group do
      // so at different times) would part ways - r02d: illegal instruction / illegal address at >= 300 envs.  The flags are only
      // read under the lock: read while another group stores them they may mix old and new values.
      int got = 0;
      if (lane == 0) {
        for (;;) {
          int old = atomicCAS(E.lock + e, 0, 1);
          if (old == 0) {
            __threadfence();
            if (env_is_busy(E, e)) got = 1;
            else atomicExch(E.lock + e, 0);
            break;
          }
          // an earlier visit of this env still runs elsewhere: it takes this visit's iterations over
          if (atomicCAS(E.lock + e, old, old + 2 * n_it) == old) break;
        }
      }
      got = group_bcast_int(got, lane);
      if (!got) continue;
      __threadfence();
      if (GE_NW > 1 && lane == 0) g_hovf = E.gws ? E.gws + (size_t)e * L.hfull : nullptr;  // this env's Hessian overflow row
      env_load(E, e, ws, lane, r);
      env = e; running = true;
      left = n_it;
    }
#if GE_NW == 1
    __syncwarp();
    if (!__syncthreads_or(env >= 0)) break;  // all warps (= envs) of the CTA are out of work
#else
    if (env < 0) break;                      // one env per CTA: `env` is the same in every thread
#endif
    if (env < 0) { stage_barriers_idle((stage_sync & 1) != 0); continue; }
    bool stepped = false;
    // one iteration of the reference loop that ends in a physics step (or the env going idle)
    while (true) {
      if (!r.c.active) {
        if (r.p.phase == PH_NONE || !prog_advance(r.p, r.c, ws, lane, base, r.info, &r.reward)) { running = false; break; }
        continue;
      }
      double delta = pid_and_delta(ws, lane, r.c.mask, c_m.timestep);
      if (delta < r.c.tol) { r.c.result = 1; r.c.reached = 1; }
      if (r.c.steps > r.c.maxsteps) { r.c.result = 2; r.c.active = 0; continue; }
      if (!(stage_sync & 0x100)) sim_step(ws, wi, lane, &r.status, (stage_sync & 1) != 0);  // bit 8: GE_DBG_NOSTEP (scheduler-only experiments)
      stepped = true;
      r.c.steps++; r.nstep++;
      if (r.c.reached) r.c.active = 0;
      break;
    }
    if (!stepped) stage_barriers_idle((stage_sync & 1) != 0);
    if (--left <= 0 || !running) {
      // a movement that just ended inside the last iteration still has to hand over to the program (no sub-step involved)
      while (!r.c.active && r.p.phase != PH_NONE) { if (!prog_advance(r.p, r.c, ws, lane, base, r.info, &r.reward)) break; }
      gsync();
      env_store(E, env, ws, lane, r);
      __threadfence();
      gsync();
      // let go of the env, or run the iterations that later visits handed over meanwhile (the state is still in shared memory)
      int more = 0;
      if (lane == 0) {
        if (!running) atomicExch(E.lock + env, 0);  // idle env: handed-over iterations have nothing to do
        else for (;;) {
          int old = atomicCAS(E.lock + env, 1, 0);
          if (old == 1) break;
          if (atomicCAS(E.lock + env, old, 1) == old) { more = old >> 1; break; }
        }
      }
      more = group_bcast_int(more, lane);
      r.nstep = 0;  // env_store added them to the env's sub-step counter
      if (more > 0) left = more;
      else env = -1;
    }
  }
}
// number of environments that still have a movement / program pending (ge_run's loop condition)
__global__ void k_count_busy(EnvArrays E, int n_env) {
  int env = blockIdx.x * blockDim.x + threadIdx.x;
  int b = env < n_env && (E.cmd_active[env] || E.prog_phase[env] != PH_NONE);
  unsigned m = __ballot_sync(FULL, b);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(E.busy_count, __popc(m));
}

// forward pipeline on one env, selected intermediate copied out (parity tests); no integration
__global__ void __launch_bounds__(GE_LANES) k_debug(EnvArrays E, int env, int field, double* out, int cap, int* nout) {
  extern __shared__ double smem[];
  const DevModel& m = c_m; const Layout& L = c_L;
  int lane = threadIdx.x;
  double* ws = smem;
  if (GE_NW > 1 && threadIdx.x == 0) g_hovf = E.gws ? E.gws + (size_t)env * L.hfull : nullptr;
  int* wi = (int*)(ws + L.total_doubles);
  LANE_LOOP(i, m.nq) ws[L.qpos + i] = E.qpos[(size_t)env * m.nq + i];
  LANE_LOOP(i, m.nv) { ws[L.qvel + i] = E.qvel[(size_t)env * m.nv + i]; ws[L.qaccws + i] = E.qaccws[(size_t)env * m.nv + i]; }
  if (lane < 32) ws[L.ctl + lane] = E.ctl[(size_t)env * 32 + lane];
  gsync();
  int status = 0, n = 0;
  if (field <= 2) {  // kinematics only: 0 xpos, 1 xmat, 2 cdof
    stage_fk(ws, lane);
    const double* src = field == 0 ? ws + L.xpos : (field == 1 ? ws + L.xmat : ws + L.cdof);
    n = field == 0 ? 3 * m.nbody : (field == 1 ? 9 * m.nbody : 6 * m.nv);
    LANE_LOOP(i, (n < cap ? n : cap)) out[i] = src[i];
  } else if (field == 3 || field == 4) {  // 3 qM (sparse), 4 qfrc_bias
    stage_fk(ws, lane); stage_rne(ws, lane);
    if (field == 4) { n = m.nv; LANE_LOOP(i, (n < cap ? n : cap)) out[i] = ws[L.qfrc_smooth + i]; }
    else { gsync(); stage_crb(ws, lane); n = m.nM; LANE_LOOP(i, (n < cap ? n : cap)) out[i] = ws[L.qM + i]; }
  } else {
    StepInfo si = forward(ws, wi, lane, &status);
    if (field == 5 || field == 6 || field == 7) {
      const double* src = field == 5 ? ws + L.qacc_smooth : (field == 6 ? ws + L.qacc : ws + L.qfrc_constraint);
      n = m.nv;
      LANE_LOOP(i, (n < cap ? n : cap)) out[i] = src[i];
    } else if (field == 8) {  // contacts: dist,pos3,frame9,geom1,geom2,dim
      n = 16 * si.ncon;
      LANE_LOOP(i, si.ncon) if (16 * i + 16 <= cap) {
        const double* c = ws + L.con + i * L.cstride;
        for (int k = 0; k < 13; k++) out[16 * i + k] = c[k];
        int p = wi[L.i_cpair + i];
        out[16 * i + 13] = m.pair_geom[2 * p]; out[16 * i + 14] = m.pair_geom[2 * p + 1]; out[16 * i + 15] = wi[L.i_cdim + i];
      }
    } else if (field == 9) { n = 1; if (lane == 0) out[0] = si.ncon; }
    else if (field == 10) { n = 1; if (lane == 0) out[0] = si.niter; }
    else if (field == 11) { n = 1; if (lane == 0) out[0] = si.nsr; }
  }
  if (lane == 0) *nout = n;
}

__global__ void k_set_state(EnvArrays E, int n_env, int nq, int nv, const double* qpos, const double* qvel, const unsigned char* mask) {
  int env = blockIdx.x * blockDim.y + threadIdx.y, lane = threadIdx.x;
  if (env >= n_env || (mask && !mask[env])) return;
  const DevModel& m = c_m;
  for (int i = lane; i < nq; i += 32) E.qpos[(size_t)env * nq + i] = qpos[(size_t)env * nq + i];
  for (int i = lane; i < nv; i += 32) { E.qvel[(size_t)env * nv + i] = qvel ? qvel[(size_t)env * nv + i] : 0.0; E.qaccws[(size_t)env * nv + i] = 0.0; }
  double* ctl = E.ctl + (size_t)env * 32;
  if (lane < GE_NU) {
    double q = qpos[(size_t)env * nq + m.jnt_qposadr[m.actuator_jntid[lane]]];
    ctl[CTL_TARGET + lane] = q; ctl[CTL_LAST + lane] = q; ctl[CTL_KP + lane] = m.pid_kp[lane]; ctl[CTL_CTRL + lane] = 0;
  } else if (lane < 8) { ctl[CTL_TARGET + lane] = ctl[CTL_LAST + lane] = ctl[CTL_KP + lane] = ctl[CTL_CTRL + lane] = 0; }
  if (lane == 0) {
    E.cmd_active[env] = 0; E.cmd_result[env] = 0; E.cmd_steps[env] = 0; E.prog_phase[env] = PH_NONE; E.reward[env] = 0; E.status[env] = 0;
    for (int k = 0; k < 12; k++) E.prog_info[12 * env + k] = 0;
  }
}
__global__ void k_set_gain(EnvArrays E, int n_env, int act, const double* kp, double value) {
  int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env < n_env) E.ctl[(size_t)env * 32 + CTL_KP + act] = kp ? kp[env] : value;
}
// kind: 0 move_group, 1 move_ee (xyz), 2 stay (aux = chunks), 3 grasp program
__global__ void k_command(EnvArrays E, int n_env, int kind, int mask, const double* target, const double* xyz, const int* rot, double tol,
                          int maxsteps, int aux, double table, const unsigned char* emask, double bx, double by, double bz) {
  int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n_env || (emask && !emask[env])) return;
  double* ctl = E.ctl + (size_t)env * 32;
  E.prog_phase[env] = PH_NONE;
  if (kind == 0) {
    if (target) for (int i = 0; i < GE_NU; i++) if (mask >> i & 1) ctl[CTL_TARGET + i] = target[(size_t)env * GE_NU + i];
    E.cmd_active[env] = 1; E.cmd_mask[env] = mask; E.cmd_tol[env] = tol; E.cmd_maxsteps[env] = maxsteps; E.cmd_steps[env] = 1; E.cmd_result[env] = 0;
  } else if (kind == 1) {
    double q5[5];
    const double base[3] = {bx, by, bz};
    if (!ik_solve(xyz + 3 * env, base, q5)) { E.cmd_active[env] = 0; E.cmd_result[env] = 3; E.cmd_steps[env] = 0; return; }
    for (int i = 0; i < 5; i++) ctl[CTL_TARGET + i] = q5[i];
    E.cmd_active[env] = 1; E.cmd_mask[env] = 0x1f; E.cmd_tol[env] = tol; E.cmd_maxsteps[env] = maxsteps; E.cmd_steps[env] = 1; E.cmd_result[env] = 0;
  } else if (kind == 2) {
    if (aux <= 0) { E.cmd_active[env] = 0; return; }
    E.prog_phase[env] = PH_STAY_ONLY; E.prog_aux[env] = aux;
    E.cmd_active[env] = 1; E.cmd_mask[env] = 0x7f; E.cmd_tol[env] = 1e-7; E.cmd_maxsteps[env] = 10; E.cmd_steps[env] = 1; E.cmd_result[env] = 0;
  } else {
    E.prog_phase[env] = PH_PRE; E.prog_rot[env] = rot[env]; E.prog_grasp[env] = 0; E.prog_aux[env] = 0; E.prog_table[env] = table;
    for (int k = 0; k < 3; k++) E.prog_coords[3 * env + k] = xyz[3 * env + k];
    for (int k = 0; k < 12; k++) E.prog_info[12 * env + k] = 0;
    E.reward[env] = 0;
    double q5[5], c1[3] = {xyz[3 * env], xyz[3 * env + 1], 1.1};
    const double base[3] = {bx, by, bz};
    if (!ik_solve(c1, base, q5)) { E.cmd_active[env] = 0; E.cmd_result[env] = 3; E.cmd_steps[env] = 0; return; }
    for (int i = 0; i < 5; i++) ctl[CTL_TARGET + i] = q5[i];
    E.cmd_active[env] = 1; E.cmd_mask[env] = 0x1f; E.cmd_tol[env] = 0.05; E.cmd_maxsteps[env] = 1000; E.cmd_steps[env] = 1; E.cmd_result[env] = 0;
  }
}
__global__ void k_targets(EnvArrays E, int n_env, const double* in, double* out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_env * GE_NU) return;
  int env = i / GE_NU, a = i % GE_NU;
  if (in) E.ctl[(size_t)env * 32 + CTL_TARGET + a] = in[i];
  if (out) out[i] = E.ctl[(size_t)env * 32 + CTL_TARGET + a];
}
// sim.data.ctrl[:] = values (MJ_Controller.actuate_joint_group, MujocoController.py:256-267) / read-back
__global__ void k_ctrl(EnvArrays E, int n_env, const double* in, double* out, const unsigned char* emask) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_env * GE_NU) return;
  int env = i / GE_NU, a = i % GE_NU;
  if (in && !(emask && !emask[env])) E.ctl[(size_t)env * 32 + CTL_CTRL + a] = in[i];
  if (out) out[i] = E.ctl[(size_t)env * 32 + CTL_CTRL + a];
}
// `nsub` bare sim.step() calls with the controls as they stand (no PID evaluation): what a caller of the reference gets from
// sim.step() after actuate_joint_group (MujocoController.py:256-267, :611).  One warp per CTA; not a throughput path.
__global__ void __launch_bounds__(GE_LANES) k_step_open(EnvArrays E, int n_env, int nsub, const unsigned char* emask) {
  extern __shared__ double smem[];
  const DevModel& m = c_m; const Layout& L = c_L;
  int env = blockIdx.x, lane = threadIdx.x;
  if (env >= n_env || (emask && !emask[env])) return;
  double* ws = smem;
  if (GE_NW > 1 && threadIdx.x == 0) g_hovf = E.gws ? E.gws + (size_t)env * L.hfull : nullptr;
  int* wi = (int*)(ws + L.total_doubles);
  LANE_LOOP(i, m.nq) ws[L.qpos + i] = E.qpos[(size_t)env * m.nq + i];
  LANE_LOOP(i, m.nv) { ws[L.qvel + i] = E.qvel[(size_t)env * m.nv + i]; ws[L.qaccws + i] = E.qaccws[(size_t)env * m.nv + i]; }
  if (lane < 32) ws[L.ctl + lane] = E.ctl[(size_t)env * 32 + lane];
  gsync();
  int status = E.status[env];
  for (int it = 0; it < nsub; it++) sim_step(ws, wi, lane, &status, false);
  LANE_LOOP(i, m.nq) E.qpos[(size_t)env * m.nq + i] = ws[L.qpos + i];
  LANE_LOOP(i, m.nv) { E.qvel[(size_t)env * m.nv + i] = ws[L.qvel + i]; E.qaccws[(size_t)env * m.nv + i] = ws[L.qaccws + i]; }
  if (lane == 0) { E.status[env] = status; E.substeps[env] += nsub; }
}
__global__ void k_busy(EnvArrays E, int n_env, unsigned char* busy) {
  int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env < n_env) busy[env] = (E.cmd_active[env] || E.prog_phase[env] != PH_NONE) ? 1 : 0;
}
__global__ void k_ik(int n, const double* xyz, double* q5, unsigned char* ok, double bx, double by, double bz) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double base[3] = {bx, by, bz};
  double q[5];
  bool r = ik_solve(xyz + 3 * i, base, q);
  for (int k = 0; k < 5; k++) q5[5 * i + k] = q[k];
  ok[i] = r;
}
// pixel_2_world (MujocoController.py:783-806): pos_w = R^-1 (K^-1 [x,y,1] * (-depth) + cam_pos)
__global__ void k_pixel_2_world(int n, int cam, int W, int H, const int* px, const int* py, const float* depth, double* xyz) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const DevModel& m = c_m;
  const double PI = 3.14159265358979323846;
  double f = 0.5 * H / tan(m.cam_fovy[cam] * PI / 360.0), d = -(double)depth[i];
  double pc[3] = {(px[i] * d - 0.5 * W * d) / f, (py[i] * d - 0.5 * H * d) / f, d}, t[3];
  v3add(t, pc, m.cam_pos0 + 3 * cam);
  m3Tmulv(xyz + 3 * i, m.cam_mat0 + 9 * cam, t);  // inverse of a rotation matrix = transpose
}
__global__ void __launch_bounds__(GE_LANES) k_body_xpos(EnvArrays E, int n_env, double* xpos) {
  extern __shared__ double smem[];
  const DevModel& m = c_m; const Layout& L = c_L;
  int env = blockIdx.x, lane = threadIdx.x;
  if (env >= n_env) return;
  double* ws = smem;
  LANE_LOOP(i, m.nq) ws[L.qpos + i] = E.qpos[(size_t)env * m.nq + i];
  gsync();
  stage_fk(ws, lane);
  LANE_LOOP(i, 3 * m.nbody) xpos[(size_t)env * 3 * m.nbody + i] = ws[L.xpos + i];
}

}  // namespace ge

// ------------------------------------------------------------------------------------------------ host side
struct BlobEntry { char name[32]; int32_t dtype, ndim; int64_t shape[4]; int64_t offset, nbytes; };

struct ge_engine {
  int device, n_envs;
  cudaStream_t stream;
  DevModel hm;       // host copy of the struct holding DEVICE pointers
  Layout lay;
  size_t ws_smem;    // dynamic shared memory per env of the stepping kernels (0: workspace in HBM)
  EnvArrays E;
  void* dblob;       // whole blob on the device
  std::vector<char> hblob;
  double base_pos[3];
  int64_t launches, substep_launches;
  int wpb;           // warps (= envs) per CTA of the sub-step kernel
  int stage_sync;    // CTA barriers between the stages of a sub-step (instruction-cache sharing)
  int quota;         // iterations per visit of k_run's dynamic env scheduling
  int max_ctas;      // resident CTAs of k_run on this device (persistent grid)
  unsigned long long ticket_base;  // tasks issued by all previous launches
  int* d_nout; double* d_dbg;
  RenderCtx rctx;
};

static const void* blob_find(const std::vector<char>& b, const char* name, int64_t* count) {
  int64_t n = *(const int64_t*)(b.data() + 8);
  const BlobEntry* e = (const BlobEntry*)(b.data() + 24);
  for (int64_t i = 0; i < n; i++)
    if (strncmp(e[i].name, name, 32) == 0) {
      int64_t c = 1;
      for (int k = 0; k < e[i].ndim; k++) c *= e[i].shape[k];
      if (count) *count = c;
      return b.data() + e[i].offset;
    }
  return nullptr;
}
static int64_t blob_off(const std::vector<char>& b, const char* name) {
  const void* p = blob_find(b, name, nullptr);
  return p ? (const char*)p - b.data() : -1;
}

struct ge_engine;
static ge_engine* g_bound = nullptr;  // engine whose model / layout currently sit in __constant__ memory

static int align_up(int x, int a) { return (x + a - 1) / a * a; }

static void make_layout(const DevModel& m, Layout& L, const int* tree_dofnum_h, const int* tree_simple_h, int ntree_dofnum_n, int maxcon, int hcap) {
  int nb = m.nbody, nj = m.njnt, nv = m.nv, ng = m.ngeom;
  int o = 0;
  auto take = [&](int n) { int r = o; o += align_up(n, 2); return r; };
  L.qpos = take(m.nq); L.qvel = take(nv); L.qaccws = take(nv); L.ctl = take(32);
  L.cdof = take(6 * nv); L.qM = take(m.nM);
  {  // the tree-sparse L^T D L factor is only needed when a tree is too wide for the lane-group mass solve
    bool need = false;
    for (int t = 0; t < ntree_dofnum_n; t++) if (tree_dofnum_h[t] > 8 && !tree_simple_h[t]) need = true;
    L.qLD = need ? take(m.nM) : L.qM;
  }
  L.qfrc_smooth = take(nv); L.qacc_smooth = take(nv); L.qfrc_constraint = take(nv); L.qacc = take(nv);
  L.Ma = take(nv); L.grad = take(nv); L.search = take(nv); L.Mv = take(nv);
  L.cstride = align_up(C_MU + 4 * m.maxdim - 1, 2);
  // list capacities: the 6-object scene never exceeded 20 contacts; piles of free objects need room for ~3 contacts per object
  L.maxcon = maxcon;
  L.maxcand = 2 * L.maxcon;
  L.con = take(L.maxcon * L.cstride);
  L.sr = take(6 * GE_MAXSR);
  L.scratch = o;
  // phase A (kinematics/dynamics/collision)
  // phase A (kinematics -> collision -> bias forces / mass matrix); order of use:
  //   stage_fk writes everything; stage_collision needs gpos/gmat/gcen only; stage_rne + stage_crb need cinert (+ their own
  //   temporaries, which overwrite the geom frames and body poses that are dead by then)
  int a = L.scratch;
  auto takeA = [&](int n) { int r = a; a += align_up(n, 2); return r; };
  L.gpos = takeA(3 * ng); L.gmat = takeA(9 * ng); L.gcen = takeA(3 * ng);  // alive until the end of collision
  L.xpos = takeA(3 * nb); L.xmat = takeA(9 * nb);                            // alive until the end of stage_fk
  L.xquat = L.xpos; L.xipos = L.xpos;                                        // (not stored any more)
  int a_local = a;
  L.lpos = takeA(3 * nb); L.lquat = takeA(4 * nb); L.janchor = takeA(3 * nj); L.jaxis = takeA(3 * nj);  // dead before cinert is written
  int endA1 = a;
  L.cinert = a_local;                                                         // alive until CRB
  if (a_local + 10 * nb > endA1) endA1 = a_local + align_up(10 * nb, 2);
  // RNE / CRB temporaries start at the scratch base (geom frames and body poses are dead after collision) and must end below cinert
  a = L.scratch;
  L.cdofdot = takeA(6 * nv); L.cvel = takeA(6 * nb); L.cacc = takeA(6 * nb); L.cfrc = takeA(6 * nb);
  int endA2 = a;
  if (endA2 > L.cinert) {  // not enough room below cinert: move cinert (and the local frames) up
    int shift = endA2 - L.cinert;
    L.cinert += shift; L.lpos += shift; L.lquat += shift; L.janchor += shift; L.jaxis += shift; endA1 += shift;
  }
  // phase B (solver)
  int b = L.scratch;
  auto takeB = [&](int n) { int r = b; b += align_up(n, 2); return r; };
  L.hfull = nv * (nv + 1) / 2;
  L.hcap = hcap > 0 && hcap < L.hfull ? hcap : L.hfull;
  L.H = takeB(L.hcap); L.Vb = takeB(6 * nb); L.Wb = takeB(6 * nb);
  int endB = b;
  // crb (10*nb) is written over cvel+cacc (12*nb) — asserted by construction (cvel, cacc adjacent)
  int end = endA1 > endA2 ? endA1 : endA2;
  if (endB > end) end = endB;
  L.total_doubles = align_up(end, 2);
  L.fk_bytes = align_up(endA1, 2) * 8;
  int io = 0;
  auto takeI = [&](int n) { int r = io; io += n; return r; };
  L.i_cb1 = takeI(L.maxcon); L.i_cb2 = takeI(L.maxcon); L.i_ct1 = takeI(L.maxcon); L.i_ct2 = takeI(L.maxcon); L.i_cdim = takeI(L.maxcon); L.i_cpair = takeI(L.maxcon); L.i_cact = takeI(L.maxcon);
  L.i_srA = takeI(GE_MAXSR); L.i_srB = takeI(GE_MAXSR); L.i_srtype = takeI(GE_MAXSR); L.i_sract = takeI(GE_MAXSR);
  L.i_cand = takeI(L.maxcand); L.i_first = takeI(nv); L.i_tcoupled = takeI(m.ntree); L.i_tcount = takeI(m.ntree); L.i_tlist = takeI(m.ntree * GE_TLIST); L.i_island = takeI(m.ntree); L.i_hflag = takeI(GE_NW > 1 ? 1 : 0);
  L.total_ints = align_up(io, 4);
  L.total_bytes = L.total_doubles * 8 + L.total_ints * 4;
  L.ws_global = 0;
}

extern "C" int ge_create(const void* model_blob, size_t nbytes, int n_envs, int device, void* stream, ge_handle* out) {
  if (!model_blob || nbytes < 32 || n_envs <= 0 || !out) return fail(GE_ERR_ARG, "ge_create: bad argument");
  if (memcmp(model_blob, "GEBLOB01", 8) != 0) return fail(GE_ERR_MODEL, "ge_create: not a model blob");
  CK(cudaSetDevice(device));
  ge_engine* h = new ge_engine();
  h->device = device; h->n_envs = n_envs; h->stream = (cudaStream_t)stream; h->launches = h->substep_launches = 0;
  h->hblob.assign((const char*)model_blob, (const char*)model_blob + nbytes);
  CK(cudaMalloc(&h->dblob, nbytes));
  CK(cudaMemcpy(h->dblob, model_blob, nbytes, cudaMemcpyHostToDevice));
  DevModel& m = h->hm;
  memset(&m, 0, sizeof m);
  const std::vector<char>& B = h->hblob;
  bool missing = false;
  auto I = [&](const char* n) -> int { const void* p = blob_find(B, n, nullptr); if (!p) { missing = true; fail(GE_ERR_MODEL, "blob entry missing: %s", n); return 0; } return *(const int32_t*)p; };
  auto D = [&](const char* n) -> double { const void* p = blob_find(B, n, nullptr); if (!p) { missing = true; fail(GE_ERR_MODEL, "blob entry missing: %s", n); return 0; } return *(const double*)p; };
  auto PD = [&](const char* n) -> const double* { int64_t o = blob_off(B, n); if (o < 0) { missing = true; fail(GE_ERR_MODEL, "blob entry missing: %s", n); return nullptr; } return (const double*)((char*)h->dblob + o); };
  auto PI = [&](const char* n) -> const int* { int64_t o = blob_off(B, n); if (o < 0) { missing = true; fail(GE_ERR_MODEL, "blob entry missing: %s", n); return nullptr; } return (const int*)((char*)h->dblob + o); };
  m.nbody = I("nbody"); m.njnt = I("njnt"); m.nq = I("nq"); m.nv = I("nv"); m.nu = I("nu"); m.ngeom = I("ngeom"); m.neq = I("neq");
  m.npair = I("npair"); m.nmesh = I("nmesh"); m.nM = I("nM"); m.ntree = I("ntree");
  m.timestep = D("opt_timestep"); m.tolerance = D("opt_tolerance"); m.impratio = D("opt_impratio"); m.mpr_tol = D("opt_mpr_tolerance");
  m.meaninertia = D("stat_meaninertia"); m.extent = D("stat_extent"); m.zfar = D("vis_zfar");
  m.iterations = I("opt_iterations"); m.mpr_iter = I("opt_mpr_iterations"); m.ik_base_body = I("ik_base_body"); m.ee_body = I("ee_body");
  { const double* g = (const double*)blob_find(B, "opt_gravity", nullptr); if (g) memcpy(m.gravity, g, 24); else missing = true; }
  m.qpos0 = PD("qpos0"); m.body_pos = PD("body_pos"); m.body_quat = PD("body_quat"); m.body_mass = PD("body_mass"); m.body_ipos = PD("body_ipos");
  m.body_inertia = PD("body_inertia"); m.body_invweight0 = PD("body_invweight0");
  m.body_parentid = PI("body_parentid"); m.body_jntadr = PI("body_jntadr"); m.body_jntnum = PI("body_jntnum"); m.body_lastdof = PI("body_lastdof");
  m.body_subtreenum = PI("body_subtreenum"); m.body_chainmask = PI("body_chainmask");
  m.jnt_type = PI("jnt_type"); m.jnt_bodyid = PI("jnt_bodyid"); m.jnt_qposadr = PI("jnt_qposadr"); m.jnt_dofadr = PI("jnt_dofadr"); m.jnt_limited = PI("jnt_limited");
  m.jnt_pos = PD("jnt_pos"); m.jnt_axis = PD("jnt_axis"); m.jnt_range = PD("jnt_range"); m.jnt_margin = PD("jnt_margin"); m.jnt_solref = PD("jnt_solref"); m.jnt_solimp = PD("jnt_solimp");
  m.dof_bodyid = PI("dof_bodyid"); m.dof_jntid = PI("dof_jntid"); m.dof_parentid = PI("dof_parentid"); m.dof_Madr = PI("dof_Madr");
  m.dof_subtreenum = PI("dof_subtreenum"); m.dof_depth = PI("dof_depth"); m.dof_treeindex = PI("dof_treeindex"); m.tree_dofadr = PI("tree_dofadr"); m.tree_dofnum = PI("tree_dofnum"); m.tree_simple = PI("tree_simple"); m.tree_Minv = PD("tree_Minv");
  m.dof_armature = PD("dof_armature"); m.dof_damping = PD("dof_damping"); m.dof_invweight0 = PD("dof_invweight0");
  m.geom_type = PI("geom_type"); m.geom_bodyid = PI("geom_bodyid"); m.geom_meshid = PI("geom_meshid");
  m.geom_pos = PD("geom_pos"); m.geom_lmat = PD("geom_lmat"); m.geom_size = PD("geom_size"); m.geom_rbound = PD("geom_rbound");
  m.geom_obbcenter = PD("geom_obbcenter"); m.geom_obbhalf = PD("geom_obbhalf"); m.geom_rgba = PD("geom_rgba");
  m.mesh_vertadr = PI("mesh_vertadr"); m.mesh_vertnum = PI("mesh_vertnum"); m.mesh_faceadr = PI("mesh_faceadr"); m.mesh_facenum = PI("mesh_facenum");
  m.mesh_vert = PD("mesh_vert"); m.mesh_center = PD("mesh_center"); m.mesh_faceplane = PD("mesh_faceplane");
  m.pair_geom = PI("pair_geom"); m.pair_rec = PI("pair_rec"); m.pair_rsum = PD("pair_rsum"); m.pair_condim = PI("pair_condim"); m.pair_friction = PD("pair_friction"); m.pair_margin = PD("pair_margin");
  m.pair_solref = PD("pair_solref"); m.pair_solimp = PD("pair_solimp");
  m.actuator_jntid = PI("actuator_jntid"); m.actuator_gear = PD("actuator_gear"); m.actuator_ctrlrange = PD("actuator_ctrlrange");
  m.eq_jnt1 = PI("eq_jnt1"); m.eq_jnt2 = PI("eq_jnt2"); m.eq_polycoef = PD("eq_polycoef"); m.eq_solref = PD("eq_solref"); m.eq_solimp = PD("eq_solimp");
  m.cam_pos0 = PD("cam_pos0"); m.cam_mat0 = PD("cam_mat0"); m.cam_fovy = PD("cam_fovy");
  m.pid_kp = PD("pid_kp"); m.pid_kd = PD("pid_kd"); m.pid_lim = PD("pid_lim");
  m.ik_chain = PD("ik_chain"); m.ik_lower = PD("ik_lower"); m.ik_upper = PD("ik_upper"); m.ik_offset = PD("ik_offset");
  if (missing) { cudaFree(h->dblob); delete h; return GE_ERR_MODEL; }
  if (m.nu != GE_NU) { cudaFree(h->dblob); delete h; return fail(GE_ERR_MODEL, "model must have 7 actuators"); }
  if (m.ntree > 64) { cudaFree(h->dblob); delete h; return fail(GE_ERR_MODEL, "model has more than 64 kinematic trees"); }
  {
    int64_t cnt = 0;
    const int32_t* cd = (const int32_t*)blob_find(B, "pair_condim", &cnt);
    m.maxdim = 1;
    for (int64_t i = 0; i < cnt; i++) if (cd[i] > m.maxdim) m.maxdim = cd[i];
    const double* damp = (const double*)blob_find(B, "dof_damping", &cnt);
    m.any_damping = 0;
    for (int64_t i = 0; i < cnt; i++) if (damp[i] != 0) m.any_damping = 1;
    const double* bp = (const double*)blob_find(B, "ik_base_pos", &cnt);
    if (!bp) { cudaFree(h->dblob); delete h; return fail(GE_ERR_MODEL, "blob entry missing: %s", "ik_base_pos"); }
    memcpy(h->base_pos, bp, 24);
  }
  const int* tdn = (const int*)blob_find(B, "tree_dofnum", nullptr);
  const int* tsi = (const int*)blob_find(B, "tree_simple", nullptr);
  // list capacities: the 6-object scene never exceeded 20 contacts; piles of free objects need room for ~3 contacts per object
  const int maxcon_default = m.ntree <= 8 ? 32 : 128;
#if GE_NW == 1
  // warp-per-env build: the whole workspace (full Hessian triangle) in one shared-memory slice per warp, or not at all
  make_layout(m, h->lay, tdn, tsi, m.ntree, maxcon_default, 0);
  h->lay.ws_global = 0;
  if (h->lay.total_bytes > 227 * 1024) { cudaFree(h->dblob); delete h; return fail(GE_ERR_TOO_LARGE, "per-env workspace exceeds shared memory"); }
#else
  // CTA-per-env build: the workspace of ONE env per CTA in shared memory.  The Hessian block region is capped so that two CTAs share
  // an SM (2 x 113 KB); a Hessian build that needs more (one huge island) uses the env's overflow row in HBM for that build.
  {
    // 112 contacts instead of the 128 of the r01 HBM layout: with 128 the phase-aliased workspace of the 40-object scene is 116.9 KB even
    // with an empty Hessian region - 3.3 KB over what lets two CTAs share an SM (settled piles hold 40-50 contacts; overflow is flagged)
    int maxcon = maxcon_default > 112 ? 112 : maxcon_default;
    if (const char* ev = getenv("GE_MAXCON")) { int v = atoi(ev); if (v >= 16 && v <= 512) maxcon = v; }
    int diag = 0;
    for (int t = 0; t < m.ntree; t++) diag += tdn[t] * (tdn[t] + 1) / 2;
    const int hfull = m.nv * (m.nv + 1) / 2;
    int need_min = diag + 6 * maxcon + 64;  // all trees uncoupled / the contact-wrench scratch of nt_update
    if (need_min > hfull) need_min = hfull;
    // the Hessian region shares the phase-aliased scratch with the kinematics arrays: largest cap whose layout fits the budget
    auto fit = [&](long budget) {
      int lo = 0, hi = hfull;  // largest cap in [1, hfull] with total_bytes <= budget (0: none)
      while (lo < hi) {
        int mid = (lo + hi + 1) / 2;
        Layout T;
        make_layout(m, T, tdn, tsi, m.ntree, maxcon, mid);
        if ((long)T.total_bytes <= budget) lo = mid; else hi = mid - 1;
      }
      return lo;
    };
    const long budget2 = 233472 / 2 - 1024 - 2048, budget1 = 227 * 1024 - 2048;  // per CTA: system reserve and the static arrays taken off
    int cap = fit(budget2);
    if (cap < need_min) cap = fit(budget1);
    if (cap < need_min) { cudaFree(h->dblob); delete h; return fail(GE_ERR_MODEL, "model too large: per-env workspace exceeds shared memory even with one CTA per SM"); }
    if (const char* ev = getenv("GE_HCAP")) { long v = atol(ev); if (v >= need_min && v <= hfull) cap = (int)v; }
    make_layout(m, h->lay, tdn, tsi, m.ntree, maxcon, cap);
    if (h->lay.total_bytes > 227 * 1024) { cudaFree(h->dblob); delete h; return fail(GE_ERR_MODEL, "model too large: per-env workspace exceeds shared memory"); }
    h->lay.ws_global = 1;
  }
#endif
  if (h->lay.fk_bytes > 227 * 1024) { cudaFree(h->dblob); delete h; return fail(GE_ERR_MODEL, "model too large: kinematics workspace exceeds shared memory"); }
  CK(cudaMemcpyToSymbol(c_m, &m, sizeof m));
  CK(cudaMemcpyToSymbol(c_L, &h->lay, sizeof(Layout)));
  { int nc = 0; if (const char* ev = getenv("GE_NANCHECK")) nc = atoi(ev) != 0; CK(cudaMemcpyToSymbol(c_nancheck, &nc, sizeof nc)); }
  // warps (= envs) per CTA: maximise the resident warps per SM (228 KB shared memory per SM, 1 KB reserved per CTA, 227 KB max per
  // CTA); ties go to the smaller CTA (less barrier imbalance).  r01 sweeps are in DESIGN.md; GE_WPB overrides.
  if (GE_NW > 1) h->wpb = 1;  // CTA-per-env build: one environment per CTA of GE_NW warps
  else {
    int best = 1, best_warps = 0;
    for (int w = 1; w <= 8; w++) {
      long per_cta = (long)w * h->lay.total_bytes;
      if (per_cta > 227 * 1024) break;
      int ctas = (int)(233472 / (per_cta + 1024));
      if (ctas > 32) ctas = 32;
      if (w * ctas > best_warps) { best_warps = w * ctas; best = w; }
    }
    h->wpb = best;
  }
  h->stage_sync = 1;  // lock-step warps of a CTA share instruction-cache lines (warp-per-env build)
  if (const char* ev = getenv("GE_STAGE_SYNC")) h->stage_sync = atoi(ev) != 0;
  if (GE_NW > 1) h->stage_sync = 0;
  if (const char* ev = getenv("GE_DBG_NOSTEP")) if (atoi(ev) != 0) h->stage_sync |= 0x100;
  if (const char* ev = getenv("GE_WPB")) if (GE_NW == 1) { int v = atoi(ev); if (v >= 1 && v <= 8 && v * h->lay.total_bytes <= 227 * 1024) h->wpb = v; }
  h->ws_smem = (size_t)h->lay.total_bytes;
  if (getenv("GE_VERBOSE"))
    fprintf(stderr, "grasp_engine: %s build, workspace %d B per env (%d doubles + %d ints), contacts <= %d, Hessian region %d of %d doubles, %d env(s) per CTA\n",
            GE_NW > 1 ? "CTA-per-env" : "warp-per-env", h->lay.total_bytes, h->lay.total_doubles, h->lay.total_ints, h->lay.maxcon, h->lay.hcap, h->lay.hfull, h->wpb);
  if (h->ws_smem) {
    CK(cudaFuncSetAttribute(k_run, cudaFuncAttributeMaxDynamicSharedMemorySize, h->wpb * h->lay.total_bytes));
    if (h->lay.total_bytes > 48 * 1024) {
      CK(cudaFuncSetAttribute(k_debug, cudaFuncAttributeMaxDynamicSharedMemorySize, h->lay.total_bytes));
      CK(cudaFuncSetAttribute(k_step_open, cudaFuncAttributeMaxDynamicSharedMemorySize, h->lay.total_bytes));
    }
  }
  if (h->lay.fk_bytes > 48 * 1024) CK(cudaFuncSetAttribute(k_body_xpos, cudaFuncAttributeMaxDynamicSharedMemorySize, h->lay.fk_bytes));
  EnvArrays& E = h->E;
  size_t N = n_envs;
#define AL(ptr, type, cnt) CK(cudaMalloc(&ptr, sizeof(type) * (cnt))); CK(cudaMemset(ptr, 0, sizeof(type) * (cnt)))
  AL(E.qpos, double, N * m.nq); AL(E.qvel, double, N * m.nv); AL(E.qaccws, double, N * m.nv); AL(E.ctl, double, N * 32);
  AL(E.cmd_mask, int, N); AL(E.cmd_maxsteps, int, N); AL(E.cmd_steps, int, N); AL(E.cmd_result, int, N); AL(E.cmd_active, int, N); AL(E.cmd_tol, double, N);
  AL(E.prog_phase, int, N); AL(E.prog_rot, int, N); AL(E.prog_grasp, int, N); AL(E.prog_aux, int, N); AL(E.prog_info, int, N * 12);
  AL(E.prog_coords, double, N * 3); AL(E.prog_table, double, N); AL(E.reward, unsigned char, N); AL(E.status, int, N); AL(E.substeps, long long, N);
  AL(E.busy_count, int, 1); AL(E.lock, int, N); AL(E.ticket, unsigned long long, 1);
  h->ticket_base = 0;
  h->quota = 32;  // r02c sweep at 4096 envs: 32 -> 3.89 M, 64 -> 3.81 M, 128 -> 3.59 M, 256 (= one visit per launch) -> 3.24 M sub-steps/s
  if (const char* ev = getenv("GE_QUOTA")) { int v = atoi(ev); if (v >= 1) h->quota = v; }
  {
    int per_sm = 0, sms = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_run, GE_LANES * h->wpb, (size_t)h->wpb * h->ws_smem));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    h->max_ctas = per_sm * sms > 0 ? per_sm * sms : 1;
    if (const char* ev = getenv("GE_MAXCTAS")) { int v = atoi(ev); if (v >= 1 && v < h->max_ctas) h->max_ctas = v; }  // experiments: fewer resident CTAs
  }
  E.gws = nullptr;
  if (h->lay.hcap < h->lay.hfull) { AL(E.gws, double, N * (size_t)h->lay.hfull); }
  AL(h->d_nout, int, 1); AL(h->d_dbg, double, 1 << 16);
#undef AL
  render_init(h->rctx, m, h->hblob.data());
  // initial state: qpos0 for every env, controller targets = current joint angles
  {
    std::vector<double> q((size_t)N * m.nq);
    const double* q0 = (const double*)blob_find(B, "qpos0", nullptr);
    for (size_t e = 0; e < N; e++) memcpy(q.data() + e * m.nq, q0, sizeof(double) * m.nq);
    double* dq;
    CK(cudaMalloc(&dq, q.size() * 8));
    CK(cudaMemcpy(dq, q.data(), q.size() * 8, cudaMemcpyHostToDevice));
    dim3 blk(32, 4);
    k_set_state<<<(n_envs + 3) / 4, blk, 0, h->stream>>>(E, n_envs, m.nq, m.nv, dq, nullptr, nullptr);
    h->launches++;
    CK(cudaStreamSynchronize(h->stream));
    cudaFree(dq);
  }
  g_bound = h;
  *out = h;
  return GE_OK;
}

extern "C" int ge_destroy(ge_handle h) {
  if (!h) return GE_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  if (g_bound == h) g_bound = nullptr;
  EnvArrays& E = h->E;
  void* ptrs[] = {E.qpos, E.qvel, E.qaccws, E.ctl, E.cmd_mask, E.cmd_maxsteps, E.cmd_steps, E.cmd_result, E.cmd_active, E.cmd_tol, E.prog_phase,
                  E.prog_rot, E.prog_grasp, E.prog_aux, E.prog_info, E.prog_coords, E.prog_table, E.reward, E.status, E.substeps, E.busy_count,
                  h->d_nout, h->d_dbg, h->dblob, E.gws, E.lock, E.ticket};
  for (void* p : ptrs) cudaFree(p);
  render_free(h->rctx);
  delete h;
  return GE_OK;
}

extern "C" int ge_size(ge_handle h, int what) {
  if (!h) return GE_ERR_ARG;
  switch (what) {
    case 0: return h->hm.nq; case 1: return h->hm.nv; case 2: return h->hm.nbody; case 3: return h->hm.ngeom; case 4: return h->hm.nu;
    case 5: return h->n_envs; case 6: return h->lay.maxcon; case 7: return h->lay.total_bytes; case 8: return h->wpb; case 9: return h->lay.ws_global;
  }
  return GE_ERR_ARG;
}

// The model / layout live in __constant__ memory of this module.  Engines of different scenes may coexist in one process:
// the constants are re-uploaded (after draining the device) whenever a call arrives for an engine other than the last one used.
static int bind(ge_handle h) {
  CK(cudaSetDevice(h->device));
  if (g_bound != h) {
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpyToSymbol(c_m, &h->hm, sizeof(DevModel)));
    CK(cudaMemcpyToSymbol(c_L, &h->lay, sizeof(Layout)));
    g_bound = h;
  }
  return GE_OK;
}

extern "C" int ge_set_state(ge_handle h, const double* qpos, const double* qvel, const uint8_t* env_mask) {
  if (!h || !qpos) return fail(GE_ERR_ARG, "ge_set_state: bad argument");
  if (bind(h)) return GE_ERR_CUDA;
  dim3 blk(32, 4);
  k_set_state<<<(h->n_envs + 3) / 4, blk, 0, h->stream>>>(h->E, h->n_envs, h->hm.nq, h->hm.nv, qpos, qvel, env_mask);
  h->launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
extern "C" int ge_get_state(ge_handle h, double* qpos, double* qvel) {
  if (!h) return GE_ERR_ARG;
  if (bind(h)) return GE_ERR_CUDA;
  if (qpos) CK(cudaMemcpyAsync(qpos, h->E.qpos, sizeof(double) * h->n_envs * h->hm.nq, cudaMemcpyDeviceToDevice, h->stream));
  if (qvel) CK(cudaMemcpyAsync(qvel, h->E.qvel, sizeof(double) * h->n_envs * h->hm.nv, cudaMemcpyDeviceToDevice, h->stream));
  return GE_OK;
}
extern "C" int ge_get_body_xpos(ge_handle h, double* xpos) {
  if (!h || !xpos) return GE_ERR_ARG;
  if (bind(h)) return GE_ERR_CUDA;
  k_body_xpos<<<h->n_envs, GE_LANES, h->lay.fk_bytes, h->stream>>>(h->E, h->n_envs, xpos);
  h->launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
extern "C" int ge_set_gain(ge_handle h, int actuator, const double* kp, double value) {
  if (!h || actuator < 0 || actuator >= GE_NU) return fail(GE_ERR_ARG, "ge_set_gain: bad actuator");
  if (bind(h)) return GE_ERR_CUDA;
  k_set_gain<<<(h->n_envs + 127) / 128, 128, 0, h->stream>>>(h->E, h->n_envs, actuator, kp, value);
  h->launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
static int command(ge_handle h, int kind, int mask, const double* target, const double* xyz, const int* rot, double tol, int maxsteps, int aux,
                   double table, const uint8_t* emask) {
  if (bind(h)) return GE_ERR_CUDA;
  k_command<<<(h->n_envs + 127) / 128, 128, 0, h->stream>>>(h->E, h->n_envs, kind, mask, target, xyz, rot, tol, maxsteps, aux, table, emask,
                                                              h->base_pos[0], h->base_pos[1], h->base_pos[2]);
  h->launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
extern "C" int ge_move_group(ge_handle h, int group_mask, const double* target, double tolerance, int max_steps, const uint8_t* env_mask) {
  if (!h || group_mask <= 0 || group_mask > 0x7f) return fail(GE_ERR_ARG, "ge_move_group: bad group mask");
  return command(h, 0, group_mask, target, nullptr, nullptr, tolerance, max_steps, 0, 0, env_mask);
}
extern "C" int ge_move_ee(ge_handle h, const double* xyz, double tolerance, int max_steps, const uint8_t* env_mask) {
  if (!h || !xyz) return fail(GE_ERR_ARG, "ge_move_ee: bad argument");
  return command(h, 1, 0x1f, nullptr, xyz, nullptr, tolerance, max_steps, 0, 0, env_mask);
}
extern "C" int ge_stay(ge_handle h, int duration_ms, const uint8_t* env_mask) {
  if (!h || duration_ms < 0) return fail(GE_ERR_ARG, "ge_stay: bad argument");
  return command(h, 2, 0x7f, nullptr, nullptr, nullptr, 1e-7, 10, (duration_ms / 2 + 9) / 10, 0, env_mask);
}
extern "C" int ge_grasp(ge_handle h, const double* coords, const int32_t* rot, double table_height, const uint8_t* env_mask) {
  if (!h || !coords || !rot) return fail(GE_ERR_ARG, "ge_grasp: bad argument");
  return command(h, 3, 0, nullptr, coords, rot, 0, 0, 0, table_height, env_mask);
}

extern "C" int ge_run_async(ge_handle h, int substeps) {
  if (!h || substeps <= 0) return fail(GE_ERR_ARG, "ge_run_async: bad argument");
  if (bind(h)) return GE_ERR_CUDA;
  dim3 blk(GE_LANES, h->wpb);
  int ctas = (h->n_envs + h->wpb - 1) / h->wpb;
  if (ctas > h->max_ctas) ctas = h->max_ctas;  // persistent grid: environments are handed to warps dynamically
  int quota = h->quota < substeps ? h->quota : substeps;
  k_run<<<ctas, blk, (size_t)h->wpb * h->ws_smem, h->stream>>>(h->E, h->n_envs, substeps, quota, h->ticket_base, h->base_pos[0], h->base_pos[1],
                                                                h->base_pos[2], h->stage_sync);
  // every warp takes tasks until it has drawn one beyond the launch's range: n_env * visits real tasks + one overshoot per warp
  h->ticket_base += (unsigned long long)h->n_envs * ((substeps + quota - 1) / quota) + (unsigned long long)ctas * h->wpb;  // (one drawing group per env slot)
  h->launches++; h->substep_launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
extern "C" int ge_run(ge_handle h, int max_substeps, int* n_busy) {
  if (!h) return GE_ERR_ARG;
  if (bind(h)) return GE_ERR_CUDA;
  const int chunk = 256;
  int done = 0, busy = 1;
  while (busy) {
    int n = chunk;
    if (max_substeps > 0) { if (done >= max_substeps) break; if (max_substeps - done < n) n = max_substeps - done; }
    CK(cudaMemsetAsync(h->E.busy_count, 0, sizeof(int), h->stream));
    int r = ge_run_async(h, n);
    if (r) return r;
    k_count_busy<<<(h->n_envs + 127) / 128, 128, 0, h->stream>>>(h->E, h->n_envs);
    h->launches++;
    CK(cudaMemcpyAsync(&busy, h->E.busy_count, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    done += n;
  }
  if (n_busy) *n_busy = busy;
  return GE_OK;
}

extern "C" int ge_get_results(ge_handle h, int32_t* result, int32_t* steps, uint8_t* reward, int64_t* total_substeps) {
  if (!h) return GE_ERR_ARG;
  if (bind(h)) return GE_ERR_CUDA;
  size_t N = h->n_envs;
  if (result) CK(cudaMemcpyAsync(result, h->E.cmd_result, 4 * N, cudaMemcpyDeviceToDevice, h->stream));
  if (steps) CK(cudaMemcpyAsync(steps, h->E.cmd_steps, 4 * N, cudaMemcpyDeviceToDevice, h->stream));
  if (reward) CK(cudaMemcpyAsync(reward, h->E.reward, N, cudaMemcpyDeviceToDevice, h->stream));
  if (total_substeps) CK(cudaMemcpyAsync(total_substeps, h->E.substeps, 8 * N, cudaMemcpyDeviceToDevice, h->stream));
  return GE_OK;
}
extern "C" int ge_get_grasp_info(ge_handle h, int32_t* info) {
  if (!h || !info) return GE_ERR_ARG;
  if (bind(h)) return GE_ERR_CUDA;
  CK(cudaMemcpyAsync(info, h->E.prog_info, 4 * 12 * (size_t)h->n_envs, cudaMemcpyDeviceToDevice, h->stream));
  return GE_OK;
}
extern "C" int ge_get_status(ge_handle h, int32_t* status) {
  if (!h || !status) return GE_ERR_ARG;
  if (bind(h)) return GE_ERR_CUDA;
  CK(cudaMemcpyAsync(status, h->E.status, 4 * (size_t)h->n_envs, cudaMemcpyDeviceToDevice, h->stream));
  return GE_OK;
}
extern "C" int ge_set_targets(ge_handle h, const double* target) {
  if (!h || !target) return GE_ERR_ARG;
  if (bind(h)) return GE_ERR_CUDA;
  k_targets<<<(h->n_envs * GE_NU + 127) / 128, 128, 0, h->stream>>>(h->E, h->n_envs, target, nullptr);
  h->launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
extern "C" int ge_get_targets(ge_handle h, double* target) {
  if (!h || !target) return GE_ERR_ARG;
  if (bind(h)) return GE_ERR_CUDA;
  k_targets<<<(h->n_envs * GE_NU + 127) / 128, 128, 0, h->stream>>>(h->E, h->n_envs, nullptr, target);
  h->launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
extern "C" int ge_set_ctrl(ge_handle h, const double* ctrl, const uint8_t* env_mask) {
  if (!h || !ctrl) return fail(GE_ERR_ARG, "ge_set_ctrl: bad argument");
  if (bind(h)) return GE_ERR_CUDA;
  k_ctrl<<<(h->n_envs * GE_NU + 127) / 128, 128, 0, h->stream>>>(h->E, h->n_envs, ctrl, nullptr, env_mask);
  h->launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
extern "C" int ge_get_ctrl(ge_handle h, double* ctrl) {
  if (!h || !ctrl) return fail(GE_ERR_ARG, "ge_get_ctrl: bad argument");
  if (bind(h)) return GE_ERR_CUDA;
  k_ctrl<<<(h->n_envs * GE_NU + 127) / 128, 128, 0, h->stream>>>(h->E, h->n_envs, nullptr, ctrl, nullptr);
  h->launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
extern "C" int ge_step_open_loop(ge_handle h, int substeps, const uint8_t* env_mask) {
  if (!h || substeps <= 0) return fail(GE_ERR_ARG, "ge_step_open_loop: bad argument");
  if (bind(h)) return GE_ERR_CUDA;
  k_step_open<<<h->n_envs, GE_LANES, h->ws_smem, h->stream>>>(h->E, h->n_envs, substeps, env_mask);
  h->launches++; h->substep_launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
extern "C" int ge_get_busy(ge_handle h, uint8_t* busy) {
  if (!h || !busy) return GE_ERR_ARG;
  if (bind(h)) return GE_ERR_CUDA;
  k_busy<<<(h->n_envs + 127) / 128, 128, 0, h->stream>>>(h->E, h->n_envs, busy);
  h->launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
extern "C" int ge_ik(ge_handle h, const double* xyz, double* q5, uint8_t* ok) {
  if (!h || !xyz || !q5 || !ok) return GE_ERR_ARG;
  if (bind(h)) return GE_ERR_CUDA;
  k_ik<<<(h->n_envs + 127) / 128, 128, 0, h->stream>>>(h->n_envs, xyz, q5, ok, h->base_pos[0], h->base_pos[1], h->base_pos[2]);
  h->launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
extern "C" int ge_pixel_2_world(ge_handle h, int cam, int width, int height, const int32_t* px, const int32_t* py, const float* depth, double* xyz) {
  if (!h || !px || !py || !depth || !xyz) return GE_ERR_ARG;
  if (bind(h)) return GE_ERR_CUDA;
  k_pixel_2_world<<<(h->n_envs + 127) / 128, 128, 0, h->stream>>>(h->n_envs, cam, width, height, px, py, depth, xyz);
  h->launches++;
  CK(cudaGetLastError());
  return GE_OK;
}
extern "C" int ge_render(ge_handle h, int cam, int width, int height, uint8_t* rgb, float* depth_m) {
  if (!h || !rgb || !depth_m || width <= 0 || height <= 0) return fail(GE_ERR_ARG, "ge_render: bad argument");
  if (bind(h)) return GE_ERR_CUDA;
  int r = render_launch(h->rctx, h->hm, h->lay, h->E.qpos, h->n_envs, cam, width, height, rgb, depth_m, h->stream, &h->launches);
  if (r) return fail(GE_ERR_CUDA, "ge_render: %s", cudaGetErrorString(cudaGetLastError()));
  return GE_OK;
}

extern "C" int ge_debug_forward(ge_handle h, int env, const char* field, double* out, int cap) {
  if (!h || !field || !out || env < 0 || env >= h->n_envs) return fail(GE_ERR_ARG, "ge_debug_forward: bad argument");
  if (bind(h)) return GE_ERR_CUDA;
  static const char* names[] = {"xpos", "xmat", "cdof", "qM", "qfrc_bias", "qacc_smooth", "qacc", "qfrc_constraint", "contact", "ncon", "niter", "nsr"};
  int f = -1;
  for (int i = 0; i < 12; i++) if (!strcmp(names[i], field)) f = i;
  if (f < 0) return fail(GE_ERR_ARG, "ge_debug_forward: unknown field %s", field);
  if (cap > (1 << 16)) cap = 1 << 16;
  k_debug<<<1, GE_LANES, h->ws_smem, h->stream>>>(h->E, env, f, h->d_dbg, cap, h->d_nout);
  h->launches++;
  CK(cudaGetLastError());
  int n = 0;
  CK(cudaMemcpyAsync(&n, h->d_nout, 4, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (n > cap) n = cap;
  CK(cudaMemcpy(out, h->d_dbg, sizeof(double) * n, cudaMemcpyDeviceToHost));
  return n;
}
extern "C" int ge_counters(ge_handle h, int64_t* kernel_launches, int64_t* substep_launches) {
  if (!h) return GE_ERR_ARG;
  if (kernel_launches) *kernel_launches = h->launches;
  if (substep_launches) *substep_launches = h->substep_launches;
  return GE_OK;
}
