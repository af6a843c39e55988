// step_kernel.cu -- CUDA kernels + C ABI (include/uhc_b200.h) for the batched humanoid env: one warp per environment,
// working set in shared memory, state records in HBM.  sm_100a.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include "../../include/uhc_b200.h"
#ifndef UHC_EPB_F
#define UHC_EPB_F 7
#endif
#include "env_step.h"
#include "eval_internal.h"
#include "clip_table.h"

using namespace uhc;

static thread_local std::string g_err;
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { g_err = std::string(#x) + ": " + cudaGetErrorString(e_); return -1; } } while (0)

// the small per-model tables every solve walks (joint gains / armature, tree-level table) are staged once per CTA behind the
// EPB work sets; the Model is pointed at the copies (sim_core.h reads them with shared-space loads)
template <class Real, int EPB>
__device__ __forceinline__ void stage_tables(EngineView<Real> &ev, unsigned char *smem) {
    Real *s_dof = reinterpret_cast<Real *>(smem + EPB * sizeof(Work<Real>));
    Real *s_lim = s_dof + NV * 4;
    int *s_lvl = reinterpret_cast<int *>(s_lim + NV * 4);
    for (int i = threadIdx.x; i < NV * 4; i += blockDim.x) { s_dof[i] = ev.model.dof_f[i]; s_lim[i] = ev.model.dof_lim[i]; }
    for (int i = threadIdx.x; i < (MAXLEVEL + 1) * LVL_G; i += blockDim.x) s_lvl[i] = ev.model.lvl_pack[i];
    LaneTopo *s_topo = reinterpret_cast<LaneTopo *>(s_lvl + (MAXLEVEL + 1) * LVL_G);
    if (threadIdx.x < 32) s_topo[threadIdx.x] = lane_topo(ev.model, (int)threadIdx.x);
    __syncthreads();
    ev.model.dof_f = s_dof; ev.model.dof_lim = s_lim; ev.model.lvl_pack = s_lvl; ev.model.topo_s = s_topo;
}

#ifndef UHC_MIN_CTAS
#define UHC_MIN_CTAS 2
#endif
#ifdef UHC_MAXNREG     /* experiment knob: cap registers without changing the CTA shape */
#define UHC_STEP_BOUNDS(EPB, Real) __maxnreg__(UHC_MAXNREG)
#else
#define UHC_STEP_BOUNDS(EPB, Real) __launch_bounds__(32 * EPB, (sizeof(Real) == 4 && EPB <= 7 ? UHC_MIN_CTAS : 1))
#endif
// EVAL: the evaluation mode of uhc_evaluate (EvalView, env_step.h): idle slots return at once (no physics, not counted as invalid),
// active slots record their step and take the next clip of the queue in place of auto_reset.  The rollout instantiation (EVAL = false)
// never reads xv.
template <class Real, int EPB, bool EVAL = false>
__global__ void UHC_STEP_BOUNDS(EPB, Real)
k_env_step(EngineView<Real> ev, const float *__restrict__ act, float *__restrict__ obs, float *__restrict__ rew, float *__restrict__ cinfo,
           int *__restrict__ fail, int *__restrict__ end, float *__restrict__ pct, float *__restrict__ torque, const int *__restrict__ order,
           const __grid_constant__ EvalView xv) {
    extern __shared__ __align__(16) unsigned char smem[];
#ifndef UHC_SYNC_SPLIT
#define UHC_SYNC_SPLIT EPB            /* warps per alignment group (experiment knob; measured: the whole CTA is best) */
#endif
    __shared__ int s_nvalid[8];
    const int warp = threadIdx.x >> 5, slot = blockIdx.x * EPB + warp, grp = warp / (UHC_SYNC_SPLIT);
    if (threadIdx.x < 8) s_nvalid[threadIdx.x] = 0;
    stage_tables<Real, EPB>(ev, smem);
    // the warps of a CTA wait for each other every substep: `order` groups environments that needed a similar number of solver
    // iterations in the previous step into the same CTA (k_order_envs), outputs stay indexed by the environment id
    const int env = slot < ev.num_envs ? (order ? order[slot] : slot) : -1;
    const bool idle = EVAL && env >= 0 && xv.slot_clip[env] < 0;
    const bool valid = env >= 0 && !idle && env_record_valid(ev, env);
    if (valid && (threadIdx.x & 31) == 0) atomicAdd(&s_nvalid[grp], 1);
    __syncthreads();
    if (!valid) {   // no work (grid tail) or a stale / never-reset env record: flagged outputs, and the warp is not counted in the substep barrier
        if (env >= 0 && !idle) env_step_invalid<Real, float>(ev, obs ? obs + (size_t)env * ev.cfg.obs_dim : nullptr, rew ? rew + env : nullptr, cinfo ? cinfo + (size_t)env * 5 : nullptr,
                                                    fail ? fail + env : nullptr, end ? end + env : nullptr, pct ? pct + env : nullptr);
        return;
    }
    Work<Real> &w = reinterpret_cast<Work<Real> *>(smem)[warp];
    if ((threadIdx.x & 31) == 0) { w.sync_threads = 32 * s_nvalid[grp]; w.sync_id = 1 + grp; }
    state_mbar_init(w);            // mbarrier of this warp's bulk-async (TMA) state load
    env_step_warp<Real, float, EVAL>(ev, env, w, act + (size_t)env * ev.cfg.act_dim, obs ? obs + (size_t)env * ev.cfg.obs_dim : nullptr, rew ? rew + env : nullptr,
                                     cinfo ? cinfo + (size_t)env * 5 : nullptr, fail ? fail + env : nullptr, end ? end + env : nullptr,
                                     pct ? pct + env : nullptr, torque ? torque + (size_t)env * NSUB * NU : nullptr, &xv);
}

// counting sort of the environments by the Newton iterations of their previous step (one block)
__global__ void __launch_bounds__(1024) k_order_envs(const int *__restrict__ istate, int E, int *__restrict__ order) {
    __shared__ int hist[64], base[64];
    if (threadIdx.x < 64) hist[threadIdx.x] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < E; i += blockDim.x) { int k = istate[(size_t)i * SI_SIZE + SI_NEWTON]; k = k < 0 ? 0 : (k > 63 ? 63 : k); atomicAdd(&hist[k], 1); }
    __syncthreads();
    if (threadIdx.x == 0) { int run = 0; for (int k = 0; k < 64; k++) { base[k] = run; run += hist[k]; } }
    __syncthreads();
    for (int i = threadIdx.x; i < E; i += blockDim.x) { int k = istate[(size_t)i * SI_SIZE + SI_NEWTON]; k = k < 0 ? 0 : (k > 63 ? 63 : k); order[atomicAdd(&base[k], 1)] = i; }
}

template <class Real, int EPB>
__global__ void __launch_bounds__(32 * EPB)
k_env_reset(EngineView<Real> ev, int n, const int *__restrict__ ids, const int *__restrict__ clip, const int *__restrict__ start,
            const int *__restrict__ len, const float *__restrict__ qpos, const float *__restrict__ qvel, float *__restrict__ obs) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int warp = threadIdx.x >> 5, i = blockIdx.x * EPB + warp;
    stage_tables<Real, EPB>(ev, smem);
    if (i >= n) return;
    Work<Real> &w = reinterpret_cast<Work<Real> *>(smem)[warp];
    const int env = ids[i];
    // optional overrides arrive as float; stage them through the work set's scratch vectors
    Real *qo = nullptr, *vo = nullptr;
    if (qpos) { qo = w.as_; vo = w.Mp; const int lane = threadIdx.x & 31;   // vectors untouched before the reset copies them out
        for (int k = lane; k < NQ; k += 32) qo[k] = (Real)qpos[(size_t)i * NQ + k];
        for (int k = lane; k < NV; k += 32) vo[k] = qvel ? (Real)qvel[(size_t)i * NV + k] : Real(0);
        __syncwarp(); }
    env_reset_warp<Real, float>(ev, env, w, clip[i], start[i], len[i], qo, vo, obs ? obs + (size_t)env * ev.cfg.obs_dim : nullptr);
}

// parity / evaluation hook: gather q, v, xpos, bquat (+ the integer record) of the listed envs into one staging array
template <class Real>
__global__ void k_gather_state(const Real *__restrict__ state, const int *__restrict__ istate, const int *__restrict__ ids, int n, double *__restrict__ out, int *__restrict__ iout) {
    const int i = blockIdx.x; if (i >= n) return;
    const int env = ids[i];
    const Real *st = state + (size_t)env * ST_SIZE;
    double *o = out + (size_t)i * 319;
    for (int k = threadIdx.x; k < NQ; k += blockDim.x) o[k] = (double)st[ST_Q + k];
    for (int k = threadIdx.x; k < NV; k += blockDim.x) o[76 + k] = (double)st[ST_V + k];
    for (int k = threadIdx.x; k < 72; k += blockDim.x) o[151 + k] = (double)st[ST_XPOS + k];
    for (int k = threadIdx.x; k < 96; k += blockDim.x) o[223 + k] = (double)st[ST_BQUAT + k];
    if (threadIdx.x < SI_SIZE) iout[(size_t)i * SI_SIZE + threadIdx.x] = istate[(size_t)env * SI_SIZE + threadIdx.x];
}
// set_state keeps cur_t and the body quaternions of the env (humanoid_im.py:902-905 only overwrites qpos / qvel)
template <class Real>
__global__ void k_save_restore_bquat(Real *__restrict__ state, int *__restrict__ istate, const int *__restrict__ ids, int n, Real *__restrict__ keep, int *__restrict__ keep_t, int restore) {
    const int i = blockIdx.x; if (i >= n) return;
    const int env = ids[i];
    Real *st = state + (size_t)env * ST_SIZE + ST_BQUAT;
    for (int k = threadIdx.x; k < 192; k += blockDim.x) { if (restore) st[k] = keep[(size_t)i * 192 + k]; else keep[(size_t)i * 192 + k] = st[k]; }
    if (threadIdx.x == 0) { if (restore) istate[(size_t)env * SI_SIZE + SI_CUR_T] = keep_t[i]; else keep_t[i] = istate[(size_t)env * SI_SIZE + SI_CUR_T]; }
}

struct UhcEngine {
    int E, device, precision, launches;
    std::vector<void *> allocs;
    EngineView<float> evf; EngineView<double> evd;
    int *d_clip_model = nullptr; int nshape = 1;
    void *d_expert = nullptr, *d_shape = nullptr; int *d_clip_adr = nullptr; float *d_clip_cdf = nullptr; int num_clips = 0;
    // staging for the host-buffer API
    float *d_act = nullptr, *d_obs = nullptr, *d_rew = nullptr, *d_cinfo = nullptr, *d_pct = nullptr; int *d_fail = nullptr, *d_end = nullptr;
    int *d_ids = nullptr; int ids_cap = 0;
    int *h_ids = nullptr;                 // pinned host staging of the reset arguments (ids, clip, start, len)
    cudaEvent_t ids_done = nullptr;       // the last reset kernel that read d_ids has been enqueued before this event
    float *d_qv = nullptr; int qv_cap = 0; void *d_keep = nullptr; int *d_keep_t = nullptr;   // set_state staging: [n][76+75] floats, kept bquat / cur_t
    double *d_gather = nullptr; int *d_gather_i = nullptr; int gather_cap = 0;
    std::vector<float> clip_w;            // clip sampling weights behind clip_cdf (uhc_set_clip_weights), empty = sample_keys rule
    int *d_order = nullptr;   // warp slot -> environment (work-sorted each step), null = identity
    std::vector<int> clip_len_h;   // host copy of the clip lengths (argument validation)
    std::vector<double> kin_h;     // [nshape][24][6] body offsets and centres of mass, fp64 (the device motion library's FK)
    std::vector<int> kin_i;        // parent [24], end-effector bodies [5]
};

template <class T> static int dev_copy(UhcEngine *e, T **dst, const T *src, size_t n) {
    CK(cudaMalloc((void **)dst, n * sizeof(T))); e->allocs.push_back(*dst);
    CK(cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice));
    return 0;
}
template <class Real> static int dev_copy_real(UhcEngine *e, const Real **dst, const double *src, size_t n) {
    std::vector<Real> tmp(n); for (size_t i = 0; i < n; i++) tmp[i] = (Real)src[i];
    Real *d; if (dev_copy(e, &d, tmp.data(), n)) return -1; *dst = d; return 0;
}
template <class Real> static void fill_cfg(EnvCfg<Real> &c, const UhcEnvCfg *h) {
    for (int i = 0; i < 4; i++) c.base_rot[i] = (Real)h->base_rot[i];
    c.rfc_scale = (Real)h->rfc_scale; c.rfc_lim = (Real)h->rfc_lim; c.rfc_rate = (Real)h->rfc_rate; c.body_diff_thresh = (Real)h->body_diff_thresh;
    c.meta_pd = h->meta_pd; c.env_episode_len = h->env_episode_len; c.trail_steps = h->trail_steps; c.newton_max_iter = h->newton_max_iter;
    for (int i = 0; i < 5; i++) { c.w[i] = (Real)h->w[i]; c.k[i] = (Real)h->k[i]; }
    c.newton_tol = (Real)h->newton_tol;
    c.auto_reset = h->auto_reset; c.t_min = h->t_min; c.t_max = h->t_max; c.reset_seed = h->reset_seed;
    c.reactive_v = h->reactive_v; c.reactive_rate = (Real)h->reactive_rate;
    c.rfc_mode = (h->rfc_mode == 1 || h->rfc_mode == 2) ? h->rfc_mode : 0; c.vf_dim = c.rfc_mode == 1 ? VF_BODY_DIM * NB : (c.rfc_mode == 2 ? 0 : 6); c.act_dim = NU + c.vf_dim + (h->meta_pd ? 2 * NSUB : 0);
    for (int b = 0; b < NB; b++) c.vf_slot[b] = (signed char)((h->vf_slot[b] >= 0 && h->vf_slot[b] < NB) ? h->vf_slot[b] : b);
    c.obs_v = (h->obs_v == 1 || h->obs_v == 3 || h->obs_v == 5 || h->obs_v == 6) ? h->obs_v : 2;
    c.fut_frames = h->fut_frames > 0 ? h->fut_frames : 10; c.fut_skip = h->fut_skip > 0 ? h->fut_skip : 10;     // cc_cfg.get("fut_frames", 10), get("skip", 10)
    c.has_shape = h->no_shape ? 0 : 1; c.obs_block = c.has_shape ? OBS_DIM : OBS_DIM - 17;
    c.obs_dim = c.obs_v == 1 ? OBS_DIM_V1 : (c.obs_v == 3 ? c.obs_block * c.fut_frames : c.obs_block);
    if (c.obs_v == 5 || c.obs_v == 6) c.obs_dim = (c.obs_v == 5 ? 636 : 384) + (c.has_shape ? 17 : 0);      // get_full_obs_v5 / v6
    c.term_body = (h->term_body == 1 || h->term_body == 2) ? h->term_body : 0; c.head_body = (h->head_body >= 0 && h->head_body < NB) ? h->head_body : 13;
    c.reward_mul = h->reward_mul ? 1 : 0;
}
template <class Real> static int build_view(UhcEngine *e, EngineView<Real> &ev, const UhcModelHost *m, const UhcEnvCfg *cfg) {
    Model<Real> &M = ev.model;
    const int nshape = m->nshape > 0 ? m->nshape : 1;
    if (dev_copy_real<Real>(e, &M.body_f, m->body_f, (size_t)nshape * NB * BODYF) || dev_copy_real<Real>(e, &M.dof_f, m->dof_f, NV * 4) ||
        dev_copy_real<Real>(e, &M.hull, m->hull, (size_t)nshape * m->nvert * 3)) return -1;
    M.nshape = nshape; M.nvert = m->nvert; M.topo_s = nullptr;
    {   // joint limits: without a table every hinge is unlimited
        std::vector<double> lim(NV * 4, 0.0);
        for (int i = 0; i < NV; i++) { lim[4 * i] = -1e30; lim[4 * i + 1] = 1e30; lim[4 * i + 2] = 1.0; }
        if (dev_copy_real<Real>(e, &M.dof_lim, m->dof_lim ? m->dof_lim : lim.data(), NV * 4)) return -1;
    }
    int *p;
#define CPI(field, n) do { if (dev_copy(e, &p, m->field, (size_t)(n))) return -1; M.field = p; } while (0)
    CPI(hull_adr, NB); CPI(hull_num, NB); CPI(nbr, m->nnbr); CPI(nbradr, m->nvert + 1); CPI(parent, NB); CPI(depth, NB); CPI(child_adr, NB + 1);
    CPI(child, NB - 1); CPI(body_sub_end, NB); CPI(ee, 5); CPI(lvl_tab, (MAXLEVEL + 1) * LVL_G * 5); CPI(lvl_pack, (MAXLEVEL + 1) * LVL_G);
#undef CPI
    M.dt = (Real)m->dt; M.margin = (Real)m->margin; M.mu = (Real)m->mu; M.solref0 = (Real)m->solref[0]; M.solref1 = (Real)m->solref[1];
    M.simp0 = (Real)m->solimp[0]; M.simp1 = (Real)m->solimp[1]; M.simp2 = (Real)m->solimp[2]; M.simp3 = (Real)m->solimp[3]; M.simp4 = (Real)m->solimp[4];
    M.gravz = (Real)m->gravz;
    fill_cfg(ev.cfg, cfg);
    ev.num_envs = e->E;
    Real *st; CK(cudaMalloc((void **)&st, (size_t)e->E * ST_SIZE * sizeof(Real))); e->allocs.push_back(st);
    CK(cudaMemset(st, 0, (size_t)e->E * ST_SIZE * sizeof(Real)));
    int *is; CK(cudaMalloc((void **)&is, (size_t)e->E * SI_SIZE * sizeof(int))); e->allocs.push_back(is);
    CK(cudaMemset(is, 0, (size_t)e->E * SI_SIZE * sizeof(int)));
    int *cn; CK(cudaMalloc((void **)&cn, 4 * sizeof(int))); e->allocs.push_back(cn); CK(cudaMemset(cn, 0, 4 * sizeof(int)));
    ev.counters = cn; ev.neutral = nullptr;
    int *el; CK(cudaMalloc((void **)&el, (size_t)e->E * 2 * sizeof(int))); e->allocs.push_back(el); CK(cudaMemset(el, 0xFF, (size_t)e->E * 2 * sizeof(int)));
    ev.ep_log = el;
    ev.state = st; ev.istate = is; ev.expert = nullptr; ev.clip_adr = nullptr; ev.clip_shape = nullptr; ev.clip_model = nullptr; ev.clip_cdf = nullptr;
    return 0;
}

constexpr int EPB_F = UHC_EPB_F, EPB_D = 2;
template <class Real, int EPB> constexpr size_t step_smem() { return EPB * sizeof(Work<Real>) + 2 * NV * 4 * sizeof(Real) + (MAXLEVEL + 1) * LVL_G * sizeof(int) + 32 * sizeof(LaneTopo); }  // environments (warps) per block
// the fp32 step kernel is tuned for UHC_MIN_CTAS resident blocks per SM (sm_100: 228 KiB of shared memory per SM, 1 KiB reserved per block, ~1 KiB static here):
// a few hundred bytes more in Work / LaneTopo silently halve the residency (measured: 1.27 -> 0.88 M env-steps/s), so it is a compile-time error
static_assert(EPB_F != 7 || UHC_MIN_CTAS * (step_smem<float, EPB_F>() + 1024 + 1088) <= 228 * 1024, "k_env_step<float>: the work sets of UHC_MIN_CTAS blocks no longer fit one SM");

extern "C" {

const char *uhc_last_error(void) { return g_err.c_str(); }

int uhc_engine_create(const UhcModelHost *model, const UhcEnvCfg *cfg, int num_envs, int device, int precision, UhcEngine **out) {
    if (!model || !cfg || !out || num_envs <= 0 || (precision != 32 && precision != 64)) { g_err = "uhc_engine_create: bad argument"; return -2; }
    CK(cudaSetDevice(device));
    UhcEngine *e = new UhcEngine();
    e->E = num_envs; e->device = device; e->precision = precision; e->launches = 0; e->nshape = model->nshape > 0 ? model->nshape : 1;
    int rc = precision == 32 ? build_view<float>(e, e->evf, model, cfg) : build_view<double>(e, e->evd, model, cfg);
    if (rc) { delete e; return rc; }
    e->kin_h.resize((size_t)e->nshape * NB * 6);
    for (int v = 0; v < e->nshape; v++) for (int b = 0; b < NB; b++) for (int k = 0; k < 6; k++) e->kin_h[((size_t)v * NB + b) * 6 + k] = model->body_f[((size_t)v * NB + b) * BODYF + k];
    e->kin_i.assign(model->parent, model->parent + NB); e->kin_i.insert(e->kin_i.end(), model->ee, model->ee + 5);
    {   // work-sorted warp slots: opt-in (UHC_SORT_ENVS=1).  Measured at 4096 envs: 1.52 M env-steps/s sorted vs 1.57 M with the identity
        // mapping -- the previous step's iteration total does not predict the per-substep imbalance well enough to pay for itself
        const char *se = getenv("UHC_SORT_ENVS");
        if (se && se[0] == '1' && num_envs > 2 * EPB_F) { CK(cudaMalloc((void **)&e->d_order, (size_t)num_envs * sizeof(int))); e->allocs.push_back(e->d_order); }
    }
    if (precision == 32) {
        CK(cudaFuncSetAttribute(k_env_step<float, EPB_F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)step_smem<float, EPB_F>()));
        CK(cudaFuncSetAttribute(k_env_step<float, EPB_F, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)step_smem<float, EPB_F>()));
        CK(cudaFuncSetAttribute(k_env_reset<float, EPB_F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)step_smem<float, EPB_F>()));
        int resident = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, k_env_step<float, EPB_F>, 32 * EPB_F, step_smem<float, EPB_F>()));
        if (EPB_F == 7 && resident < UHC_MIN_CTAS) { g_err = "uhc_engine_create: k_env_step<float> reaches only " + std::to_string(resident) + " resident block(s) per SM (built for " + std::to_string(UHC_MIN_CTAS) + ")"; delete e; return -3; }
    } else {
        CK(cudaFuncSetAttribute(k_env_step<double, EPB_D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)step_smem<double, EPB_D>()));
        CK(cudaFuncSetAttribute(k_env_step<double, EPB_D, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)step_smem<double, EPB_D>()));
        CK(cudaFuncSetAttribute(k_env_reset<double, EPB_D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)step_smem<double, EPB_D>()));
    }
    const size_t E = num_envs;
    CK(cudaMalloc((void **)&e->d_act, E * MAX_ACT_DIM * 4)); CK(cudaMalloc((void **)&e->d_obs, E * (size_t)(precision == 32 ? e->evf.cfg.obs_dim : e->evd.cfg.obs_dim) * 4)); CK(cudaMalloc((void **)&e->d_rew, E * 4));
    CK(cudaMalloc((void **)&e->d_cinfo, E * 5 * 4)); CK(cudaMalloc((void **)&e->d_pct, E * 4)); CK(cudaMalloc((void **)&e->d_fail, E * 4)); CK(cudaMalloc((void **)&e->d_end, E * 4));
    for (void *p : {(void *)e->d_act, (void *)e->d_obs, (void *)e->d_rew, (void *)e->d_cinfo, (void *)e->d_pct, (void *)e->d_fail, (void *)e->d_end}) e->allocs.push_back(p);
    *out = e;
    return 0;
}

void uhc_engine_destroy(UhcEngine *e) {
    if (!e) return;
    cudaSetDevice(e->device);
    for (void *p : e->allocs) cudaFree(p);
    if (e->d_expert) cudaFree(e->d_expert);
    if (e->d_shape) cudaFree(e->d_shape);
    if (e->d_clip_adr) cudaFree(e->d_clip_adr);
    if (e->d_clip_cdf) cudaFree(e->d_clip_cdf);
    if (e->d_clip_model) cudaFree(e->d_clip_model);
    if (e->d_ids) cudaFree(e->d_ids);
    if (e->h_ids) cudaFreeHost(e->h_ids);
    if (e->ids_done) cudaEventDestroy(e->ids_done);
    if (e->d_qv) cudaFree(e->d_qv);
    if (e->d_keep) cudaFree(e->d_keep);
    if (e->d_keep_t) cudaFree(e->d_keep_t);
    if (e->d_gather) cudaFree(e->d_gather);
    if (e->d_gather_i) cudaFree(e->d_gather_i);
    delete e;
}

// cumulative clip sampling weights: explicit weights (uhc_set_clip_weights) or the sample_keys rule of the reference
// (len // t_max + 1 copies per clip, dataset_amass_single.py:138-142)
static int upload_clip_cdf(UhcEngine *e) {
    const int nclips = e->num_clips;
    if (nclips <= 0) return 0;
    const int tmax = e->precision == 32 ? e->evf.cfg.t_max : e->evd.cfg.t_max;
    std::vector<float> cdf(nclips); double acc = 0.0;
    for (int i = 0; i < nclips; i++) {
        acc += e->clip_w.empty() ? (double)(tmax > 0 ? e->clip_len_h[i] / tmax + 1 : 1) : (double)e->clip_w[i];
        cdf[i] = (float)acc;
    }
    if (!e->d_clip_cdf) CK(cudaMalloc((void **)&e->d_clip_cdf, nclips * sizeof(float)));
    CK(cudaMemcpy(e->d_clip_cdf, cdf.data(), nclips * sizeof(float), cudaMemcpyHostToDevice));
    e->evf.clip_cdf = e->d_clip_cdf; e->evd.clip_cdf = e->d_clip_cdf;
    return 0;
}

int uhc_engine_set_cfg(UhcEngine *e, const UhcEnvCfg *cfg) {
    if (!e || !cfg) { g_err = "uhc_engine_set_cfg: null"; return -2; }
    CK(cudaSetDevice(e->device));
    const int old_tmax = e->precision == 32 ? e->evf.cfg.t_max : e->evd.cfg.t_max;
    const int old_obs_dim = uhc_engine_obs_dim(e);
    if (e->precision == 32) { fill_cfg(e->evf.cfg, cfg); e->evf.cfg.num_clips = e->num_clips; } else { fill_cfg(e->evd.cfg, cfg); e->evd.cfg.num_clips = e->num_clips; }
    if (uhc_engine_obs_dim(e) != old_obs_dim) { g_err = "uhc_engine_set_cfg: the observation width cannot change on a live engine (buffers are sized at creation)"; return -2; }
    if (cfg->t_max != old_tmax && e->clip_w.empty()) { CK(cudaDeviceSynchronize()); return upload_clip_cdf(e); }   // the sample_keys weights depend on t_max
    return 0;
}

int uhc_load_clips(UhcEngine *e, int nclips, const int *clip_len, const double *frames_host, const double *shape_host) {
    if (!e || nclips <= 0 || !clip_len || !frames_host || !shape_host) { g_err = "uhc_load_clips: bad argument"; return -2; }
    CK(cudaSetDevice(e->device));
    CK(cudaDeviceSynchronize());
    size_t total = 0;
    for (int i = 0; i < nclips; i++) { if (clip_len[i] < 2) { g_err = "uhc_load_clips: clip shorter than 2 frames"; return -2; } total += clip_len[i]; }
    const size_t nf = total * EX_SIZE, ns = (size_t)nclips * 17;
    void *d_expert = nullptr, *d_shape = nullptr;
    if (e->precision == 32) {
        std::vector<float> f(nf), s(ns);
        for (size_t i = 0; i < nf; i++) f[i] = (float)frames_host[i];
        for (size_t i = 0; i < ns; i++) s[i] = (float)shape_host[i];
        CK(cudaMalloc(&d_expert, nf * 4)); CK(cudaMalloc(&d_shape, ns * 4));
        CK(cudaMemcpy(d_expert, f.data(), nf * 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(d_shape, s.data(), ns * 4, cudaMemcpyHostToDevice));
    } else {
        CK(cudaMalloc(&d_expert, nf * 8)); CK(cudaMalloc(&d_shape, ns * 8));
        CK(cudaMemcpy(d_expert, frames_host, nf * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(d_shape, shape_host, ns * 8, cudaMemcpyHostToDevice));
    }
    return uhc_engine_install_clips(e, nclips, clip_len, d_expert, d_shape);
}

int uhc_set_neutral_pose(UhcEngine *e, const double *qpos76, const double *qvel75) {
    if (!e || !qpos76 || !qvel75) { g_err = "uhc_set_neutral_pose: bad argument"; return -2; }
    CK(cudaSetDevice(e->device));
    CK(cudaDeviceSynchronize());
    std::vector<double> h(NQ + NV);
    memcpy(h.data(), qpos76, NQ * 8); memcpy(h.data() + NQ, qvel75, NV * 8);
    if (e->precision == 32) { const float *d; if (dev_copy_real<float>(e, &d, h.data(), NQ + NV)) return -1; e->evf.neutral = d; }
    else { const double *d; if (dev_copy_real<double>(e, &d, h.data(), NQ + NV)) return -1; e->evd.neutral = d; }
    return 0;
}

int uhc_set_clip_weights(UhcEngine *e, int nclips, const float *weights_host) {
    if (!e || nclips != e->num_clips) { g_err = "uhc_set_clip_weights: call after uhc_load_clips with one weight per clip"; return -2; }
    CK(cudaSetDevice(e->device));
    if (!weights_host) e->clip_w.clear();
    else {
        double tot = 0; for (int i = 0; i < nclips; i++) { if (!(weights_host[i] >= 0.f)) { g_err = "uhc_set_clip_weights: negative / NaN weight"; return -2; } tot += weights_host[i]; }
        if (!(tot > 0)) { g_err = "uhc_set_clip_weights: all weights are zero"; return -2; }
        e->clip_w.assign(weights_host, weights_host + nclips);
    }
    CK(cudaDeviceSynchronize());
    return upload_clip_cdf(e);
}

int uhc_set_clip_models(UhcEngine *e, int nclips, const int *clip_model) {
    if (!e || !clip_model || nclips != e->num_clips) { g_err = "uhc_set_clip_models: call after uhc_load_clips with one entry per clip"; return -2; }
    for (int i = 0; i < nclips; i++) if (clip_model[i] < 0 || clip_model[i] >= e->nshape) { g_err = "uhc_set_clip_models: shape index out of range"; return -2; }
    CK(cudaSetDevice(e->device));
    if (e->d_clip_model) cudaFree(e->d_clip_model);
    CK(cudaMalloc((void **)&e->d_clip_model, nclips * sizeof(int)));
    CK(cudaMemcpy(e->d_clip_model, clip_model, nclips * sizeof(int), cudaMemcpyHostToDevice));
    e->evf.clip_model = e->d_clip_model; e->evd.clip_model = e->d_clip_model;
    return 0;
}

// no_auto_reset: the launch sees auto_reset = 0 whatever the engine's configuration (evaluation: no reactive standing-neutral starts)
static int env_reset_impl(UhcEngine *e, int n, const int *env_ids_host, const int *clip_host, const int *start_host, const int *len_host,
                          const float *qpos_dev, const float *qvel_dev, float *obs_dev, void *stream, bool no_auto_reset) {
    if (!e || n <= 0 || !env_ids_host || !clip_host || !start_host || !len_host) { g_err = "uhc_env_reset: bad argument"; return -2; }
    if (!e->d_expert) { g_err = "uhc_env_reset: no clips loaded"; return -3; }
    CK(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    for (int i = 0; i < n; i++) {
        if (env_ids_host[i] < 0 || env_ids_host[i] >= e->E) { g_err = "uhc_env_reset: env id out of range"; return -2; }
        const int c = clip_host[i];
        if (c < 0 || c >= e->num_clips) { g_err = "uhc_env_reset: clip index out of range"; return -2; }
        if (start_host[i] < 0 || len_host[i] < 1 || start_host[i] + len_host[i] > e->clip_len_h[c]) { g_err = "uhc_env_reset: (start, length) outside the clip"; return -2; }
    }
    // the arguments travel through a pinned staging buffer owned by the engine, so the caller's arrays are free on return and the
    // call stays asynchronous: the only wait is for the PREVIOUS reset's kernel to have consumed the staging buffer
    if (!e->ids_done) CK(cudaEventCreateWithFlags(&e->ids_done, cudaEventDisableTiming));
    else CK(cudaEventSynchronize(e->ids_done));
    if (e->ids_cap < n) {
        if (e->d_ids) cudaFree(e->d_ids);
        if (e->h_ids) cudaFreeHost(e->h_ids);
        const int cap = n > 256 ? n : 256;
        CK(cudaMalloc((void **)&e->d_ids, (size_t)4 * cap * sizeof(int))); CK(cudaHostAlloc((void **)&e->h_ids, (size_t)4 * cap * sizeof(int), cudaHostAllocDefault));
        e->ids_cap = cap;
    }
    memcpy(e->h_ids, env_ids_host, n * sizeof(int)); memcpy(e->h_ids + n, clip_host, n * sizeof(int));
    memcpy(e->h_ids + 2 * n, start_host, n * sizeof(int)); memcpy(e->h_ids + 3 * n, len_host, n * sizeof(int));
    CK(cudaMemcpyAsync(e->d_ids, e->h_ids, (size_t)4 * n * sizeof(int), cudaMemcpyHostToDevice, st));
    EngineView<float> evf = e->evf; EngineView<double> evd = e->evd;
    if (no_auto_reset) { evf.cfg.auto_reset = 0; evd.cfg.auto_reset = 0; }
    if (e->precision == 32)
        k_env_reset<float, EPB_F><<<(n + EPB_F - 1) / EPB_F, 32 * EPB_F, step_smem<float, EPB_F>(), st>>>(evf, n, e->d_ids, e->d_ids + n, e->d_ids + 2 * n, e->d_ids + 3 * n, qpos_dev, qvel_dev, obs_dev);
    else
        k_env_reset<double, EPB_D><<<(n + EPB_D - 1) / EPB_D, 32 * EPB_D, step_smem<double, EPB_D>(), st>>>(evd, n, e->d_ids, e->d_ids + n, e->d_ids + 2 * n, e->d_ids + 3 * n, qpos_dev, qvel_dev, obs_dev);
    CK(cudaGetLastError());
    CK(cudaEventRecord(e->ids_done, st));
    e->launches++;
    return 0;
}
int uhc_env_reset(UhcEngine *e, int n, const int *env_ids_host, const int *clip_host, const int *start_host, const int *len_host,
                  const float *qpos_dev, const float *qvel_dev, float *obs_dev, void *stream) {
    return env_reset_impl(e, n, env_ids_host, clip_host, start_host, len_host, qpos_dev, qvel_dev, obs_dev, stream, false);
}

int uhc_env_step(UhcEngine *e, const float *actions_dev, float *obs_dev, float *reward_dev, float *cinfo_dev, int *fail_dev, int *end_dev,
                 float *percent_dev, float *torque_dev, void *stream) {
    if (!e || !actions_dev) { g_err = "uhc_env_step: bad argument"; return -2; }
    if (!e->d_expert) { g_err = "uhc_env_step: no clips loaded"; return -3; }
    CK(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (e->d_order) { k_order_envs<<<1, 1024, 0, st>>>(e->precision == 32 ? e->evf.istate : e->evd.istate, e->E, e->d_order); e->launches++; }
    if (e->precision == 32)
        k_env_step<float, EPB_F><<<(e->E + EPB_F - 1) / EPB_F, 32 * EPB_F, step_smem<float, EPB_F>(), st>>>(e->evf, actions_dev, obs_dev, reward_dev, cinfo_dev, fail_dev, end_dev, percent_dev, torque_dev, e->d_order, EvalView{});
    else
        k_env_step<double, EPB_D><<<(e->E + EPB_D - 1) / EPB_D, 32 * EPB_D, step_smem<double, EPB_D>(), st>>>(e->evd, actions_dev, obs_dev, reward_dev, cinfo_dev, fail_dev, end_dev, percent_dev, torque_dev, e->d_order, EvalView{});
    CK(cudaGetLastError());
    e->launches++;
    return 0;
}

int uhc_env_step_host(UhcEngine *e, const float *actions_host, float *obs_host, float *reward_host, float *cinfo_host, int *fail_host,
                      int *end_host, float *percent_host) {
    if (!e || !actions_host) { g_err = "uhc_env_step_host: bad argument"; return -2; }
    CK(cudaSetDevice(e->device));
    const size_t E = e->E;
    CK(cudaMemcpyAsync(e->d_act, actions_host, E * (size_t)uhc_engine_act_dim(e) * 4, cudaMemcpyHostToDevice, 0));
    int rc = uhc_env_step(e, e->d_act, e->d_obs, e->d_rew, e->d_cinfo, e->d_fail, e->d_end, e->d_pct, nullptr, nullptr);
    if (rc) return rc;
    if (obs_host) CK(cudaMemcpyAsync(obs_host, e->d_obs, E * (size_t)uhc_engine_obs_dim(e) * 4, cudaMemcpyDeviceToHost, 0));
    if (reward_host) CK(cudaMemcpyAsync(reward_host, e->d_rew, E * 4, cudaMemcpyDeviceToHost, 0));
    if (cinfo_host) CK(cudaMemcpyAsync(cinfo_host, e->d_cinfo, E * 5 * 4, cudaMemcpyDeviceToHost, 0));
    if (fail_host) CK(cudaMemcpyAsync(fail_host, e->d_fail, E * 4, cudaMemcpyDeviceToHost, 0));
    if (end_host) CK(cudaMemcpyAsync(end_host, e->d_end, E * 4, cudaMemcpyDeviceToHost, 0));
    if (percent_host) CK(cudaMemcpyAsync(percent_host, e->d_pct, E * 4, cudaMemcpyDeviceToHost, 0));
    CK(cudaStreamSynchronize(0));
    return 0;
}

// state of n envs in one gather kernel + one copy: out = [n][319] doubles (qpos76 qvel75 xpos72 bquat96), iout = [n][8]
int uhc_env_get_state_batch(UhcEngine *e, int n, const int *env_ids_host, double *out_host, int *istate_host) {
    if (!e || n <= 0 || !env_ids_host || !out_host) { g_err = "uhc_env_get_state_batch: bad argument"; return -2; }
    for (int i = 0; i < n; i++) if (env_ids_host[i] < 0 || env_ids_host[i] >= e->E) { g_err = "uhc_env_get_state_batch: env id out of range"; return -2; }
    CK(cudaSetDevice(e->device));
    CK(cudaDeviceSynchronize());
    if (e->gather_cap < n) {
        if (e->d_gather) { cudaFree(e->d_gather); cudaFree(e->d_gather_i); }
        CK(cudaMalloc((void **)&e->d_gather, (size_t)n * 319 * sizeof(double))); CK(cudaMalloc((void **)&e->d_gather_i, (size_t)n * (SI_SIZE + 1) * sizeof(int)));
        e->gather_cap = n;
    }
    int *d_idl = e->d_gather_i + (size_t)n * SI_SIZE;
    CK(cudaMemcpy(d_idl, env_ids_host, n * sizeof(int), cudaMemcpyHostToDevice));
    if (e->precision == 32) k_gather_state<float><<<n, 128>>>(e->evf.state, e->evf.istate, d_idl, n, e->d_gather, e->d_gather_i);
    else k_gather_state<double><<<n, 128>>>(e->evd.state, e->evd.istate, d_idl, n, e->d_gather, e->d_gather_i);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out_host, e->d_gather, (size_t)n * 319 * sizeof(double), cudaMemcpyDeviceToHost));
    if (istate_host) CK(cudaMemcpy(istate_host, e->d_gather_i, (size_t)n * SI_SIZE * sizeof(int), cudaMemcpyDeviceToHost));
    return 0;
}

int uhc_env_get_state(UhcEngine *e, int env, double *qpos76, double *qvel75, double *xpos72, double *bquat96, int *istate8) {
    if (!e || env < 0 || env >= e->E) { g_err = "uhc_env_get_state: bad argument"; return -2; }
    double out[319]; int is[SI_SIZE];
    int rc = uhc_env_get_state_batch(e, 1, &env, out, is);
    if (rc) return rc;
    if (qpos76) memcpy(qpos76, out, NQ * 8);
    if (qvel75) memcpy(qvel75, out + 76, NV * 8);
    if (xpos72) memcpy(xpos72, out + 151, 72 * 8);
    if (bquat96) memcpy(bquat96, out + 223, 96 * 8);
    if (istate8) memcpy(istate8, is, sizeof is);
    return 0;
}

// fail_safe (humanoid_im.py:902-905) for n envs at once: overwrite qpos/qvel, run sim.forward(), keep cur_t and the body quats.
// One reset-with-override launch for all of them; no allocation in the steady state.
int uhc_env_set_state_batch(UhcEngine *e, int n, const int *env_ids_host, const double *qpos_host, const double *qvel_host) {
    if (!e || n <= 0 || !env_ids_host || !qpos_host || !qvel_host) { g_err = "uhc_env_set_state_batch: bad argument"; return -2; }
    for (int i = 0; i < n; i++) if (env_ids_host[i] < 0 || env_ids_host[i] >= e->E) { g_err = "uhc_env_set_state_batch: env id out of range"; return -2; }
    CK(cudaSetDevice(e->device));
    CK(cudaDeviceSynchronize());
    const size_t rs = e->precision == 32 ? 4 : 8;
    if (e->qv_cap < n) {
        if (e->d_qv) { cudaFree(e->d_qv); cudaFree(e->d_keep); cudaFree(e->d_keep_t); }
        CK(cudaMalloc((void **)&e->d_qv, (size_t)n * (NQ + NV) * 4)); CK(cudaMalloc(&e->d_keep, (size_t)n * 192 * 8)); CK(cudaMalloc((void **)&e->d_keep_t, (size_t)n * 2 * sizeof(int)));
        e->qv_cap = n;
    }
    (void)rs;
    std::vector<float> qv((size_t)n * (NQ + NV));
    for (int i = 0; i < n; i++) { for (int k = 0; k < NQ; k++) qv[(size_t)i * NQ + k] = (float)qpos_host[(size_t)i * NQ + k]; for (int k = 0; k < NV; k++) qv[(size_t)n * NQ + (size_t)i * NV + k] = (float)qvel_host[(size_t)i * NV + k]; }
    CK(cudaMemcpy(e->d_qv, qv.data(), qv.size() * 4, cudaMemcpyHostToDevice));
    std::vector<int> is((size_t)n * SI_SIZE), clip(n), start(n), len(n);
    std::vector<double> tmp((size_t)n * 319);
    int rc = uhc_env_get_state_batch(e, n, env_ids_host, tmp.data(), is.data());
    if (rc) return rc;
    for (int i = 0; i < n; i++) {
        clip[i] = is[(size_t)i * SI_SIZE + SI_CLIP]; start[i] = is[(size_t)i * SI_SIZE + SI_START]; len[i] = is[(size_t)i * SI_SIZE + SI_LEN];
        if (len[i] < 2 || clip[i] < 0 || clip[i] >= e->num_clips) { g_err = "uhc_env_set_state_batch: env has no valid episode (reset it first)"; return -2; }
    }
    int *d_idl = e->d_keep_t + n;
    CK(cudaMemcpy(d_idl, env_ids_host, n * sizeof(int), cudaMemcpyHostToDevice));
    if (e->precision == 32) k_save_restore_bquat<float><<<n, 64>>>(e->evf.state, e->evf.istate, d_idl, n, (float *)e->d_keep, e->d_keep_t, 0);
    else k_save_restore_bquat<double><<<n, 64>>>(e->evd.state, e->evd.istate, d_idl, n, (double *)e->d_keep, e->d_keep_t, 0);
    rc = uhc_env_reset(e, n, env_ids_host, clip.data(), start.data(), len.data(), e->d_qv, e->d_qv + (size_t)n * NQ, nullptr, nullptr);
    if (rc) return rc;
    if (e->precision == 32) k_save_restore_bquat<float><<<n, 64>>>(e->evf.state, e->evf.istate, d_idl, n, (float *)e->d_keep, e->d_keep_t, 1);
    else k_save_restore_bquat<double><<<n, 64>>>(e->evd.state, e->evd.istate, d_idl, n, (double *)e->d_keep, e->d_keep_t, 1);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    return 0;
}

int uhc_env_set_state(UhcEngine *e, int env, const double *qpos76, const double *qvel75) {
    return uhc_env_set_state_batch(e, 1, &env, qpos76, qvel75);
}

// device counters: out[0] = env-steps failed because a body's contacts did not fit the work set (MAXCON), out[1] = env-steps
// skipped on an invalid (stale / never reset) env record
int uhc_engine_counters(UhcEngine *e, int *out4) {
    if (!e || !out4) { g_err = "uhc_engine_counters: bad argument"; return -2; }
    CK(cudaSetDevice(e->device));
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(out4, e->precision == 32 ? e->evf.counters : e->evd.counters, 4 * sizeof(int), cudaMemcpyDeviceToHost));
    return 0;
}

const int *uhc_episode_log_dev(const UhcEngine *e) { return e ? (e->precision == 32 ? e->evf.ep_log : e->evd.ep_log) : nullptr; }
int uhc_num_envs(const UhcEngine *e) { return e ? e->E : -1; }
int uhc_engine_obs_dim(const UhcEngine *e) { return e ? (e->precision == 32 ? e->evf.cfg.obs_dim : e->evd.cfg.obs_dim) : -1; }
int uhc_engine_act_dim(const UhcEngine *e) { return e ? (e->precision == 32 ? e->evf.cfg.act_dim : e->evd.cfg.act_dim) : -1; }
int uhc_kernel_launches(const UhcEngine *e) { return e ? e->launches : -1; }

}  // extern "C"

// ---- internal entry points of the evaluation loop (eval_internal.h)
int uhc_env_step_eval(UhcEngine *e, const float *actions_dev, float *obs_dev, float *reward_dev, int *fail_dev, int *end_dev, const EvalView &xv, cudaStream_t st) {
    CK(cudaSetDevice(e->device));
    // evaluation never re-seeds by sampling: the reactive standing-neutral starts of a training reset stay off (they need auto_reset)
    if (e->precision == 32) {
        EngineView<float> ev = e->evf; ev.cfg.auto_reset = 0;
        k_env_step<float, EPB_F, true><<<(e->E + EPB_F - 1) / EPB_F, 32 * EPB_F, step_smem<float, EPB_F>(), st>>>(ev, actions_dev, obs_dev, reward_dev, e->d_cinfo, fail_dev, end_dev, e->d_pct, nullptr, nullptr, xv);
    } else {
        EngineView<double> ev = e->evd; ev.cfg.auto_reset = 0;
        k_env_step<double, EPB_D, true><<<(e->E + EPB_D - 1) / EPB_D, 32 * EPB_D, step_smem<double, EPB_D>(), st>>>(ev, actions_dev, obs_dev, reward_dev, e->d_cinfo, fail_dev, end_dev, e->d_pct, nullptr, nullptr, xv);
    }
    CK(cudaGetLastError());
    e->launches++;
    return 0;
}

int uhc_env_reset_eval(UhcEngine *e, int n, const int *env_ids_host, const int *clip_host, const int *start_host, const int *len_host, float *obs_dev,
                       cudaStream_t st) {
    return env_reset_impl(e, n, env_ids_host, clip_host, start_host, len_host, nullptr, nullptr, obs_dev, st, true);
}

int uhc_engine_expert_table(const UhcEngine *e, EngineTable *out) {
    if (!e->d_expert) { g_err = "no clips loaded"; return -3; }
    out->expert = e->d_expert; out->clip_adr = e->d_clip_adr; out->precision = e->precision; out->num_clips = e->num_clips; out->device = e->device;
    out->clip_len = e->clip_len_h.data();
    out->trail_steps = e->precision == 32 ? e->evf.cfg.trail_steps : e->evd.cfg.trail_steps;
    return 0;
}

int uhc_engine_install_clips(UhcEngine *e, int nclips, const int *clip_len, void *expert_dev, void *shape_dev) {
    CK(cudaSetDevice(e->device));
    CK(cudaDeviceSynchronize());      // in-flight work may still read the old table
    std::vector<int> adr(nclips + 1, 0);
    for (int i = 0; i < nclips; i++) adr[i + 1] = adr[i] + clip_len[i];
    if (e->d_expert) { cudaFree(e->d_expert); cudaFree(e->d_shape); cudaFree(e->d_clip_adr); cudaFree(e->d_clip_cdf); e->d_expert = e->d_shape = nullptr; e->d_clip_adr = nullptr; e->d_clip_cdf = nullptr; }
    e->d_expert = expert_dev; e->d_shape = shape_dev;
    CK(cudaMalloc((void **)&e->d_clip_adr, (nclips + 1) * sizeof(int)));
    CK(cudaMemcpy(e->d_clip_adr, adr.data(), (nclips + 1) * sizeof(int), cudaMemcpyHostToDevice));
    e->num_clips = nclips; e->clip_len_h.assign(clip_len, clip_len + nclips); e->clip_w.clear();
    e->evf.cfg.num_clips = nclips; e->evd.cfg.num_clips = nclips;
    if (upload_clip_cdf(e)) return -1;
    if (e->d_clip_model) { cudaFree(e->d_clip_model); e->d_clip_model = nullptr; }
    e->evf.clip_model = nullptr; e->evd.clip_model = nullptr;
    // every env record points into the OLD clip table: invalidate them all (len = 0); the step kernel skips (and flags) an env
    // until uhc_env_reset gives it a slice of the new table
    CK(cudaMemset(e->precision == 32 ? e->evf.istate : e->evd.istate, 0, (size_t)e->E * SI_SIZE * sizeof(int)));
    if (e->precision == 32) { e->evf.expert = (const float *)e->d_expert; e->evf.clip_shape = (const float *)e->d_shape; e->evf.clip_adr = e->d_clip_adr; }
    else { e->evd.expert = (const double *)e->d_expert; e->evd.clip_shape = (const double *)e->d_shape; e->evd.clip_adr = e->d_clip_adr; }
    return 0;
}

int uhc_engine_kin(const UhcEngine *e, EngineKin *out) {
    out->off_ipos = e->kin_h.data(); out->parent = e->kin_i.data(); out->ee = e->kin_i.data() + NB;
    out->nshape = e->nshape; out->precision = e->precision; out->device = e->device;
    return 0;
}

void uhc_engine_set_error(const char *msg) { g_err = msg; }
