// env_step.h -- one warp advances one humanoid environment by one 30 Hz control step (15 physics substeps) and runs the
// imitation-task epilogue; also the reset path.  Shared by the CUDA kernels (step_kernel.cu) and the host emulation
// (tests/emu).  Reference: uhc/envs/humanoid_im.py:1192-1243 (step), :1145-1190 (do_simulation), :1245-1299 (reset_model),
// uhc/khrylib/rl/envs/common/mujoco_env.py:95-113 (reset / set_state).
#pragma once
#include "sim_core.h"

namespace uhc {

// everything a warp needs to find its environment's data
template <class Real>
struct EngineView {
    Model<Real> model;
    EnvCfg<Real> cfg;
    int num_envs;
    Real *state;            // [E][ST_SIZE]
    int *istate;            // [E][SI_SIZE]
    const Real *expert;     // [total_frames][EX_SIZE]
    const int *clip_adr;    // [C+1] first frame of each clip in `expert`
    const Real *clip_shape; // [C][17] beta[16], gender
    const int *clip_model;  // [C] body-shape (model variant) of each clip: the reference rebuilds the robot per clip (humanoid_im.py:154-180)
    const float *clip_cdf;  // [C] cumulative sampling weights (len // t_max + 1 copies per clip, sample_keys of the reference)
    const Real *neutral;    // [76 + 75] standing_neutral qpos / qvel (sample_data/standing_neutral.pkl; humanoid_im.py:66,86), null = reactive starts off
    int *ep_log;            // [E][2] per env: clip index of the episode that ended in the last step (-1: none ended) and its completed fraction (float bits)
                            //   -- the training loop's per-clip success history (agent_copycat.py:561) is built from it
    int *counters;          // [4] device counters: 0 = env-steps failed because a body's contacts did not fit MAXCON, 1 = env-steps skipped on an invalid env record
};

// evaluation mode of the step kernel (uhc_evaluate, eval.cu): a work queue of clips [clip0, clip0 + n) over the env slots.  Slot e
// imitates clip clip0 + slot_clip[e] from frame 0 (-1: idle, no physics); every step of an active slot is recorded into row
// frame_off[i] + slot_k[e] of the per-frame outputs; a finished slot takes the next clip from queue[0] or goes idle (queue[1] counts the
// active slots).
struct EvalView {
    int clip0, n, fail_safe, reserved;
    const int *frame_off;           // [n+1]
    float *pred_qpos, *pred_jpos;   // [F][76], [F][72]
    int *frame_t;                   // [F]
    int *nframes, *last_t, *fail_any;   // [n]
    double *reward_sum;             // [n]
    int *slot_clip, *slot_k;        // [E]
    int *queue;                     // [2]
};

// an env record the step kernel can run: a clip of the CURRENT clip table and at least two frames (uhc_load_clips invalidates every
// record; never-reset envs have len = 0)
template <class Real>
UHC_DEV bool env_record_valid(const EngineView<Real> &ev, int env) {
    const int *is = ev.istate + (size_t)env * SI_SIZE;
    const int clip = is[SI_CLIP], len = is[SI_LEN];
    return len >= 2 && clip >= 0 && clip < ev.cfg.num_clips;
}
// outputs of an env that cannot be stepped: fail = end = 1, zero observation / reward (the caller must reset it)
template <class Real, class ObsT>
UHC_DEV void env_step_invalid(const EngineView<Real> &ev, ObsT *obs, ObsT *reward, ObsT *cinfo_out, int *fail_out, int *end_out, ObsT *percent_out) {
    LANES_BEGIN
    if (obs) for (int i = lane; i < ev.cfg.obs_dim; i += 32) obs[i] = (ObsT)0;
    if (cinfo_out && lane < 5) cinfo_out[lane] = (ObsT)0;
    if (lane == 0) {
        if (reward) *reward = (ObsT)0;
        if (fail_out) *fail_out = 1;
        if (end_out) *end_out = 1;
        if (percent_out) *percent_out = (ObsT)0;
#ifndef UHC_EMU
        if (ev.counters) atomicAdd(ev.counters + 1, 1);
#endif
    }
    LANES_END
}

template <class Real>
UHC_DEV const Real *expert_frame(const EngineView<Real> &ev, int clip, int start, int len, int t) {  // humanoid_im.py:1322
    // the reference slices the clip to [start, start+len) and always runs with start_ind = 0 (dataset_amass_single.py:238-244)
    const int i = start + (t < len - 1 ? t : len - 1);
    return ev.expert + (size_t)(UHC_LDG(ev.clip_adr + clip) + i) * EX_SIZE;
}

UHC_DEV unsigned long long mix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull; x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull; x = (x ^ (x >> 27)) * 0x94D049BB133111EBull; return x ^ (x >> 31);
}
// DatasetAMASSSingle.sample_seq / get_sample_from_key (dataset_amass_single.py:172-253): clip ~ sample_keys (uniform over
// len // t_max + 1 copies per clip), start ~ U{0 .. len - t_min - 1}, slice length min(t_max, len - start)
template <class Real>
UHC_DEV void sample_clip(const EngineView<Real> &ev, int env, int episode, int *clip, int *start, int *len) {
    const unsigned long long h = mix64(ev.cfg.reset_seed ^ mix64((unsigned long long)env * 0x100000001B3ull + (unsigned long long)episode));
    const float u1 = (float)(h >> 40) * (1.0f / 16777216.0f), u2 = (float)(h & 0xFFFFFF) * (1.0f / 16777216.0f);
    int lo = 0, hi = ev.cfg.num_clips - 1;
    const float target = u1 * UHC_LDG(ev.clip_cdf + hi);
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (UHC_LDG(ev.clip_cdf + mid) > target) hi = mid; else lo = mid + 1; }
    const int L = UHC_LDG(ev.clip_adr + lo + 1) - UHC_LDG(ev.clip_adr + lo);
    int span = L - ev.cfg.t_min; if (span < 1) span = 1;
    int st = (int)(u2 * (float)span); if (st > span - 1) st = span - 1;
    int ln = L - st; if (ev.cfg.t_max > 0 && ln > ev.cfg.t_max) ln = ev.cfg.t_max;
    *clip = lo; *start = st; *len = ln;
}

// model tables of the body shape a clip was recorded with
template <class Real>
UHC_DEV Model<Real> model_for_clip(const EngineView<Real> &ev, int clip) {
    Model<Real> m = ev.model;
    const int sh = ev.clip_model ? UHC_LDG(ev.clip_model + clip) : 0;
    m.body_f += (size_t)sh * NB * BODYF;
    m.hull += (size_t)sh * m.nvert * 3;
    return m;
}

// get_obs (humanoid_im.py:269-288): obs v1 / v2 against the expert frame t_next, or v3 = the v2 block repeated for fut_frames future frames
// t_next + i * skip (:505-513; expert_frame clamps past the end of the slice like get_expert_index)
template <class Real, class ObsT>
UHC_DEV void write_obs(const EngineView<Real> &ev, const Work<Real> &w, int clip, int start, int len, int t_next, ObsT *obs) {
    const Real *shape = ev.clip_shape + 17 * clip;
    if (w.cfg.obs_v == 5 || w.cfg.obs_v == 6) obs_v56(w.cfg, w, expert_frame(ev, clip, start, len, t_next), shape, obs);
    else if (w.cfg.obs_v == 3) {
        for (int f = 0; f < w.cfg.fut_frames; ++f) obs_v2(w.cfg, w, expert_frame(ev, clip, start, len, t_next + f * w.cfg.fut_skip), shape, obs + (size_t)f * w.cfg.obs_block);
    } else obs_v2(w.cfg, w, expert_frame(ev, clip, start, len, t_next), shape, obs);
}

// ---- state record <-> work set.  GPU: the head block (q v aw C Ib S, ST_BLOCK Reals) travels as ONE bulk-async copy (TMA engine:
// cp.async.bulk global -> shared completing on this warp's mbarrier; shared -> global as a bulk group), the pose arrays as 16-byte
// vector stores.  Host emulation: plain copies.
#ifndef UHC_EMU
UHC_DEV unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
template <class Real>
UHC_DEV void state_mbar_init(Work<Real> &w) {
    if ((threadIdx.x & 31) == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&w.mbar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
}
// 16-byte vector copy of n Reals (n * sizeof(Real) a multiple of 16, both sides 16-byte aligned), all lanes
template <class Real>
UHC_DEV void copy16(Real *dst, const Real *src, int n) {
    const int nv = n * (int)sizeof(Real) / 16;
    for (int i = threadIdx.x & 31; i < nv; i += 32) reinterpret_cast<uint4 *>(dst)[i] = reinterpret_cast<const uint4 *>(src)[i];
}
#endif
template <class Real>
UHC_DEV void load_state(const EngineView<Real> &ev, int env, Work<Real> &w, int parity) {
    const Real *st = ev.state + (size_t)env * ST_SIZE;
#ifndef UHC_EMU
    constexpr unsigned BYTES = ST_BLOCK * sizeof(Real);
    static_assert(BYTES % 16 == 0 && (ST_SIZE * sizeof(Real)) % 16 == 0, "bulk copies need 16-byte granularity");
    const unsigned mb = smem_u32(&w.mbar);
    if ((threadIdx.x & 31) == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mb), "r"(BYTES) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"(smem_u32(w.q)), "l"(st), "r"(BYTES), "r"(mb) : "memory");
    }
    unsigned done = 0;
    while (!done) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(done) : "r"(mb), "r"(parity) : "memory");
    }
    __syncwarp();
#else
    (void)parity;
    { Real *head = reinterpret_cast<Real *>(&w); for (int i = 0; i < ST_BLOCK; i++) head[i] = st[i]; }       // q v aw C Ib S are contiguous in Work exactly as in the record
#endif
}
template <class Real>
UHC_DEV void store_state(const EngineView<Real> &ev, int env, Work<Real> &w) {
    Real *st = ev.state + (size_t)env * ST_SIZE;
#ifndef UHC_EMU
    constexpr unsigned BYTES = ST_BLOCK * sizeof(Real);
    __syncwarp();
    copy16(st + ST_XPOS, &w.xpos[0][0], 72); copy16(st + ST_XIPOS, &w.xipos[0][0], 72); copy16(st + ST_XQUAT, &w.xquat[0][0], 96);
    if ((threadIdx.x & 31) == 0) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // the warp's generic-proxy writes to the head block -> visible to the async proxy
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(st), "r"(smem_u32(w.q)), "r"(BYTES) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");         // complete (not just read): the record may be re-read / re-written right after (in-kernel reset)
    }
    __syncwarp();
#else
    { const Real *head = reinterpret_cast<const Real *>(&w); for (int i = 0; i < ST_BLOCK; i++) st[i] = head[i]; }
    for (int i = 0; i < 72; i++) { st[ST_XPOS + i] = (&w.xpos[0][0])[i]; st[ST_XIPOS + i] = (&w.xipos[0][0])[i]; }
    for (int i = 0; i < 96; i++) st[ST_XQUAT + i] = (&w.xquat[0][0])[i];
#endif
}

// reset one env onto frame 0 of (clip, start, len): state <- expert qpos/qvel (or the override), sim.forward(), obs.
// bquat is left at the qpos0 value (identity quats) exactly as reset_model leaves it (humanoid_im.py:1277 runs before set_state).
// RESEAT: the fail-safe re-seat of uhc_env_set_state_batch (humanoid_im.py:902-905): qpos / qvel overridden, cur_t and the body
// quaternions (bquat, prev_bquat) of the running episode kept
template <class Real, class ObsT, bool RESEAT = false>
UHC_DEV void env_reset_warp(const EngineView<Real> &ev, int env, Work<Real> &w, int clip, int start, int len,
                            const Real *qpos_override, const Real *qvel_override, ObsT *obs) {
    const Real *e0 = expert_frame(ev, clip, start, len, 0);
    LANES_BEGIN
    for (int i = lane; i < NQ; i += 32) w.q[i] = qpos_override ? qpos_override[i] : e0[EX_QPOS + i];
    for (int i = lane; i < NV; i += 32) { w.v[i] = qvel_override ? qvel_override[i] : e0[EX_QVEL + i]; w.aw[i] = 0; }
    for (int i = lane; i < ACT_DIM; i += 32) w.act[i] = 0;
    LANES_END
    // reactive_v = 1, train mode (humanoid_im.py:1255-1271): with probability reactive_rate the episode starts from the standing-neutral pose,
    // turned to the expert's heading and moved to its x, y (match_heading_and_pos, :1312-1320), with the neutral velocities
    if (ev.cfg.reactive_v == 1 && ev.cfg.auto_reset && !qpos_override && ev.neutral) {
        const unsigned long long h = mix64(ev.cfg.reset_seed ^ mix64(0x5EAC71FEull + (unsigned long long)env * 0x100000001B3ull + (unsigned long long)(ev.istate[(size_t)env * SI_SIZE + SI_EPISODE] + 1)));
        if ((Real)((float)(h >> 40) * (1.0f / 16777216.0f)) < ev.cfg.reactive_rate) {
            Real q1[4], hq[4], nq[4], nh[4], nhi[4], dq[4], out[4];
            remove_base_rot(ev.cfg, e0 + EX_QPOS + 3, q1); heading_q(q1, hq);                        // heading of the expert's first frame
            for (int i = 0; i < 4; i++) nq[i] = ev.neutral[3 + i];
            heading_q(nq, nh); qinv(nh, nhi); qmul(nhi, nq, dq);                                      // de_heading of the neutral root quaternion (as stored: no base-rotation removal, :1317)
            qmul(hq, dq, out);
            LANES_BEGIN
            for (int i = lane; i < NQ; i += 32) w.q[i] = i < 2 ? e0[EX_QPOS + i] : (i >= 3 && i < 7 ? out[i - 3] : ev.neutral[i]);
            for (int i = lane; i < NV; i += 32) w.v[i] = ev.neutral[NQ + i];
            LANES_END
        }
    }
    LANES_BEGIN
    if (lane == 0) { w.mdl = model_for_clip(ev, clip); w.cfg = ev.cfg; w.con_overflow = 0; }
    LANES_END
    const Model<Real> &mdl = w.mdl;
    TOPO_DECL(mdl);
    const int iters = substep_dynamics<Real, ObsT>(mdl, w.cfg, w, tp, (const Real *)nullptr, 0, false, (ObsT *)nullptr);
    world_quat(mdl, w.q, w);
    int *is = ev.istate + (size_t)env * SI_SIZE;
    Real *st = ev.state + (size_t)env * ST_SIZE;
    LANES_BEGIN
    if constexpr (!RESEAT) for (int i = lane; i < 96; i += 32) { const Real v = (i & 3) == 0 ? Real(1) : Real(0); st[ST_BQUAT + i] = v; st[ST_PBQUAT + i] = v; }
    if (lane == 0) { if constexpr (!RESEAT) is[SI_CUR_T] = 0; is[SI_CLIP] = clip; is[SI_START] = start; is[SI_LEN] = len; is[SI_NEWTON] = iters; is[SI_NCON] = w.ncon; }
    LANES_END
    if (obs) write_obs(ev, w, clip, start, len, 1, obs);
    LANES_BEGIN
    for (int i = lane; i < NV; i += 32) w.aw[i] = 0;
    LANES_END
    store_state(ev, env, w);
}

// evaluation epilogue of an active slot (EvalView): record the step, then fail-safe re-seat, or hand the slot the next clip of the queue
template <class Real, class ObsT>
UHC_DEV void eval_after_step(const EngineView<Real> &ev, const EvalView &xv, int env, Work<Real> &w, int cur_t, int fail, int end, Real rew, ObsT *obs) {
    int *is = ev.istate + (size_t)env * SI_SIZE;
    const int i = xv.slot_clip[env], k = xv.slot_k[env];
    const int row = xv.frame_off[i] + k;
    if (row < xv.frame_off[i + 1]) {       // the caller's table holds len - 1 + trail_steps rows per clip: always true
        LANES_BEGIN
        for (int j = lane; j < NQ; j += 32) xv.pred_qpos[(size_t)row * NQ + j] = (float)w.q[j];
        for (int j = lane; j < 72; j += 32) xv.pred_jpos[(size_t)row * 72 + j] = (float)(&w.xpos[0][0])[j];     // the stored xpos (get_states)
        if (lane == 0) {
            xv.frame_t[row] = cur_t; xv.nframes[i] = k + 1; xv.last_t[i] = cur_t;
            xv.reward_sum[i] += (double)(ObsT)rew;
            if (fail) xv.fail_any[i] = 1;
        }
        LANES_END
    }
    if (!end && !(fail && !xv.fail_safe)) {
        if (fail) {   // fail_safe: the expert pose at min(cur_t, len - 1), sim.forward(); the step's own observation stays the next input
            const int clip = is[SI_CLIP], start = is[SI_START], len = is[SI_LEN];
            const Real *ef = expert_frame(ev, clip, start, len, cur_t);
            const Real *qo = ef + EX_QPOS, *vo = ef + EX_QVEL;
            if constexpr (sizeof(Real) != sizeof(float)) {   // uhc_env_set_state_batch passes the pose as float: stage it rounded, as k_env_reset does
                Real *q = w.as_, *v = w.Mp;
                LANES_BEGIN
                for (int j = lane; j < NQ; j += 32) q[j] = (Real)(float)qo[j];
                for (int j = lane; j < NV; j += 32) v[j] = (Real)(float)vo[j];
                LANES_END
                qo = q; vo = v;
            }
            env_reset_warp<Real, ObsT, true>(ev, env, w, clip, start, len, qo, vo, (ObsT *)nullptr);
        }
        LANES_BEGIN
        if (lane == 0) xv.slot_k[env] = k + 1;
        LANES_END
        return;
    }
    int j;      // the episode ended: next clip of the queue, or idle
#ifndef UHC_EMU
    j = (threadIdx.x & 31) == 0 ? atomicAdd(xv.queue, 1) : 0;
    j = __shfl_sync(0xffffffffu, j, 0);
#else
    j = xv.queue[0]++;
#endif
    if (j < xv.n) {
        const int c = xv.clip0 + j;
        env_reset_warp<Real, ObsT>(ev, env, w, c, 0, UHC_LDG(ev.clip_adr + c + 1) - UHC_LDG(ev.clip_adr + c), (const Real *)nullptr, (const Real *)nullptr, obs);
    }
    LANES_BEGIN
    if (lane == 0) {
        xv.slot_clip[env] = j < xv.n ? j : -1; xv.slot_k[env] = 0;
#ifndef UHC_EMU
        if (j >= xv.n) atomicSub(xv.queue + 1, 1);
#else
        if (j >= xv.n) xv.queue[1]--;
#endif
    }
    LANES_END
}

// one control step.  out_* may be null.  Returns done; fills flags.  EVAL: the evaluation epilogue (xv) replaces auto_reset.
template <class Real, class ObsT, bool EVAL = false>
UHC_DEV int env_step_warp(const EngineView<Real> &ev, int env, Work<Real> &w, const ObsT *action, ObsT *obs, ObsT *reward,
                          ObsT *cinfo_out, int *fail_out, int *end_out, ObsT *percent_out, ObsT *torque_out, const EvalView *xv = nullptr) {
    int *is = ev.istate + (size_t)env * SI_SIZE;
    Real *st = ev.state + (size_t)env * ST_SIZE;
    const int clip = is[SI_CLIP], start = is[SI_START], len = is[SI_LEN];
    int cur_t = is[SI_CUR_T];
    load_state(ev, env, w, 0);     // the warp's mbarrier completes exactly one phase per kernel launch
    // action = [NU joint targets | vf_dim residual-force dims | 30 meta-PD scales]: the work set keeps the joint targets, the implicit root
    // wrench and the meta-PD scales at the fixed slots the PD code reads; the explicit per-body forces are read from global memory where used
    const bool explicit_rf = ev.cfg.rfc_mode == 1;
    LANES_BEGIN
    for (int i = lane; i < NU; i += 32) w.act[i] = (Real)action[i];
    if (lane < 6) w.act[NU + lane] = ev.cfg.rfc_mode == 0 ? (Real)action[NU + lane] : Real(0);
    if (lane < 2 * NSUB) w.act[NU + 6 + lane] = ev.cfg.meta_pd ? (Real)action[NU + ev.cfg.vf_dim + lane] : Real(0);
    LANES_END
    if (explicit_rf) restore_stale_pose(w, st + ST_XPOS, st + ST_XQUAT);
    const Real *target = expert_frame(ev, clip, start, len, cur_t + 1) + EX_QPOS + 7;
    int iters = 0, maxcon = 0;
    LANES_BEGIN
    if (lane == 0) { w.mdl = model_for_clip(ev, clip); w.cfg = ev.cfg; w.con_overflow = 0; }
    LANES_END
    const Model<Real> &mdl = w.mdl;
    TOPO_DECL(mdl);
#pragma unroll 1
    for (int it = 0; it < NSUB; ++it) {
        UHC_CTA_SYNC(true);   // see substep_dynamics: the CTA's warps run each substep's straight-line code together
        iters += substep_dynamics<Real, ObsT>(mdl, w.cfg, w, tp, target, it, true, torque_out, true, action);
        if (w.ncon > maxcon) maxcon = w.ncon;
        if (it == NSUB - 1) world_quat(mdl, w.q, w);  // pose of the last forward pass (what data.body_xquat holds)
        integrate(mdl, w);
    }
    cur_t += 1;
    // body quats: prev <- stored, current from the new qpos (humanoid_im.py:1196, :1219)
    Real *bq = st + ST_BQUAT, *pbq = st + ST_PBQUAT;
    LANES_BEGIN
    for (int i = lane; i < 96; i += 32) pbq[i] = bq[i];
    LANES_END
    body_quat(w, bq);
    Real bd, rew, ci[5];
    const Real *exf = expert_frame(ev, clip, start, len, cur_t);
    diff_and_reward(mdl, w.cfg, w, exf, bq, pbq, &bd, &rew, ci, action);
    // cfg.env_term_body (humanoid_im.py:1223-1229): the mean body-position error; or the new root height / the head height of the last forward pass (data.body_xpos)
    // against the lowest of the episode's expert window - 0.1 m (expert["height_lb"], ["head_height_lb"]: tools.py:94-95 on the slice the loader handed out)
    int fail;
    if (ev.cfg.term_body == 0) fail = bd > ev.cfg.body_diff_thresh;
    else {
        const Real *f0 = ev.expert + (size_t)(UHC_LDG(ev.clip_adr + clip) + start) * EX_SIZE;
        const int off = ev.cfg.term_body == 1 ? EX_QPOS + 2 : EX_WBPOS + 3 * ev.cfg.head_body + 2;
        LVAR(Real, neg);
        LANES_BEGIN
        Real mx = Real(-1e30);
        for (int i = lane; i < len; i += 32) { const Real z = -(Real)UHC_LDG(f0 + (size_t)i * EX_SIZE + off); mx = z > mx ? z : mx; }
        LV(neg) = mx;
        LANES_END
        const Real lb = -WMAX(neg);
        fail = (ev.cfg.term_body == 1 ? w.q[2] : w.xpos[ev.cfg.head_body][2]) < lb - Real(0.1);
    }
    {   // a non-finite state can never pass "bd > thresh": flag it as a failure (mirrors the try/except at :1207-1211)
        LVAR(int, bad);
        LANES_BEGIN
        int b = 0;
        for (int i = lane; i < NQ; i += 32) if (!(w.q[i] == w.q[i]) || abs_(w.q[i]) > Real(1e6)) b = 1;
        LV(bad) = b;
        LANES_END
        if (WBALLOT(bad)) fail = 1;
    }
    // contacts that did not fit the work set: the episode is failed (and counted), never continued on a truncated contact set
    const int overflow = w.con_overflow;
    if (overflow) fail = 1;
    const int end = (cur_t >= ev.cfg.env_episode_len) || (cur_t >= len + ev.cfg.trail_steps - 1);
    if (obs) write_obs(ev, w, clip, start, len, cur_t + 1, obs);
    LANES_BEGIN
    if (lane == 0) {
        is[SI_CUR_T] = cur_t; is[SI_NEWTON] = iters; is[SI_NCON] = maxcon; is[SI_FLAGS] = overflow ? 1 : 0;
#ifndef UHC_EMU
        if (overflow && ev.counters) atomicAdd(ev.counters, 1);
#endif
        if (reward) *reward = (ObsT)rew;
        if (fail_out) *fail_out = fail;
        if (end_out) *end_out = end;
        if (percent_out) *percent_out = (ObsT)((Real)cur_t / (Real)(len - 1));
        if (ev.ep_log) {
            const float pctf = (float)((Real)cur_t / (Real)(len - 1));
            ev.ep_log[2 * env] = (fail || end) ? clip : -1;
#ifndef UHC_EMU
            ev.ep_log[2 * env + 1] = __float_as_int(pctf);
#else
            union { float f; int i; } cv; cv.f = pctf; ev.ep_log[2 * env + 1] = cv.i;
#endif
        }
    }
    if (cinfo_out && lane < 5) cinfo_out[lane] = (ObsT)ci[lane];
    LANES_END
    store_state(ev, env, w);
    if constexpr (EVAL) {
        eval_after_step<Real, ObsT>(ev, *xv, env, w, cur_t, fail, end, rew, obs);
        return fail || end;
    }
    if (ev.cfg.auto_reset && (fail || end)) {   // re-seed the finished episode in place: the next observation is the reset observation
        int nclip, nstart, nlen;
        const int episode = is[SI_EPISODE] + 1;
        sample_clip(ev, env, episode, &nclip, &nstart, &nlen);
        env_reset_warp<Real, ObsT>(ev, env, w, nclip, nstart, nlen, (const Real *)nullptr, (const Real *)nullptr, obs);
        LANES_BEGIN
        if (lane == 0) is[SI_EPISODE] = episode;
        LANES_END
    }
    return fail || end;
}

}  // namespace uhc
