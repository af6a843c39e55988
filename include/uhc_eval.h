/* uhc_eval.h -- C ABI of policy evaluation (part of libuhc_b200.so): every clip of a range imitated from frame 0 with the deterministic
 * policy, trajectories recorded and scored on the device.
 *
 * Reference interface replaced: AgentCopycat.eval_policy / eval_seq (uhc/agents/agent_copycat.py:354-494, scripts/eval_uhc.py --mode stats)
 * and the metrics of smpl_eval.compute_metrics (uhc/smpllib/smpl_eval.py:24-123; restated on the host in uhc_b200/metrics.py).
 * All pointers are CUDA device pointers owned by the caller unless suffixed _host.  Calls are stream-ordered on `stream`; return 0 on
 * success, <0 on error (uhc_eval_last_error()).
 */
#ifndef UHC_EVAL_H
#define UHC_EVAL_H
#include "uhc_b200.h"
#include "uhc_rollout.h"
#ifdef __cplusplus
extern "C" {
#endif

/* frame_metrics / clip_metrics columns, millimetres */
#define UHC_EVAL_ROOT_DIST 0
#define UHC_EVAL_MPJPE 1
#define UHC_EVAL_MPJPE_G 2
#define UHC_EVAL_PA_MPJPE 3
#define UHC_EVAL_VEL_DIST 4
#define UHC_EVAL_ACCEL_DIST 5
#define UHC_EVAL_NMETRICS 6

/* Results of uhc_evaluate for clips i = 0 .. n-1 (clip clip0 + i of the loaded table).  Clip i owns rows frame_off[i] .. frame_off[i+1]-1 of
 * the per-frame arrays, at least len_i - 1 + trail_steps of them; row frame_off[i] + k is the state after the clip's step k + 1 and rows
 * past nframes[i] are left untouched. */
typedef struct {
    const int *frame_off;      /* [n+1] */
    float *pred_qpos;          /* [F][76] qpos after the step (the "pred" trajectory) */
    float *pred_jpos;          /* [F][72] body_xpos after the step (what uhc_env_get_state returns as xpos) */
    int *frame_t;              /* [F] cur_t after the step */
    double *frame_metrics;     /* [F][6] root_dist mpjpe mpjpe_g pa_mpjpe vel_dist accel_dist; vel from a clip's 2nd row, accel from its 3rd (NaN before) */
    int *nframes, *last_t, *fail_any;   /* [n] rows recorded, cur_t of the last one, any failure on the way */
    double *reward_sum;        /* [n] sum of the step rewards */
    double *clip_metrics;      /* [n][6] per-clip means of frame_metrics (NaN where the clip has < 3 rows) */
    int frame_cap, reserved;   /* F: rows allocated behind the per-frame arrays */
} UhcEvalBuf;

const char *uhc_eval_last_error(void);

/* Evaluate clips [clip0, clip0 + n): env slot s starts on clip clip0 + s; a slot whose episode ends (clip end, or a failure without
 * fail_safe) takes the next clip of a device work queue inside the step kernel, or goes idle.  Per step: ZFilter (no update) -> policy ->
 * mean action -> physics / task; with fail_safe a failed humanoid is put back on the expert pose of frame min(cur_t, len - 1) (qpos, qvel,
 * sim.forward; cur_t and the body quaternions kept, the step's observation stays the next input), as uhc_env_set_state_batch does.  No host
 * synchronisation per step: the host reads the number of active slots every 16 steps (the step graph is captured per call, so a clip
 * table, configuration or policy changed between calls is always seen).  Then the metric stage (uhc_eval_metrics) against the
 * expert frames min(frame_t, len - 1).  Uses the engine's env records (re-seat them with uhc_env_reset afterwards); the engine's
 * auto_reset setting, and with it the reactive standing-neutral starts, is ignored during the call, for the first clip of a slot as for
 * the later ones. */
int uhc_evaluate(UhcEngine *e, int clip0, int n, const UhcMlp *mlp, const float *log_std, const double *zfilter_stats, float zclip,
                 int fail_safe, const UhcEvalBuf *out, void *stream);
int uhc_evaluate_mcp(UhcEngine *e, int clip0, int n, const UhcMcp *mcp, const float *log_std, const double *zfilter_stats, float zclip,
                     int fail_safe, const UhcEvalBuf *out, void *stream);
/* control steps of the last uhc_evaluate on this engine that started with at least one active slot (the idle steps that finish the last
 * 16-step replay are not counted) */
int uhc_eval_last_steps(UhcEngine *e, long long *steps_host);

/* the metric stage alone, fp64: n recorded trajectories, clip i in rows frame_off[i] .. frame_off[i] + nframes[i] - 1 (nframes may be NULL:
 * up to frame_off[i+1]); pred / gt qpos [F][76] and joint positions [F][72].  Fills frame_metrics [F][6] and clip_metrics [n][6] as above. */
int uhc_eval_metrics(const double *pred_qpos, const double *gt_qpos, const double *pred_jpos, const double *gt_jpos, const int *frame_off,
                     const int *nframes, int n, double *frame_metrics, double *clip_metrics, void *stream);

void uhc_eval_release(UhcEngine *e);   /* frees the evaluation scratch of this engine; call before uhc_engine_destroy */

#ifdef __cplusplus
}
#endif
#endif
