/* uhc_motion.h -- expert tables built on the device from raw SMPL pose sequences (libuhc_b200.so).
 *
 * uhc_load_clips (uhc_b200.h) takes ready-made expert records, computed on the host by uhc_b200/motion_lib.py make_expert (smpl_to_qpose +
 * Humanoid.qpos_fk of the reference, uhc/smpllib/smpl_mujoco.py:543-607, uhc/smpllib/torch_smpl_humanoid.py:155-261) and packed as
 * [frames][UHC_EX_SIZE] doubles.  uhc_load_clips_smpl computes the same records on the device, one thread per frame in fp64, from the
 * axis-angle rows and root translations alone, and writes them straight into the engine's table (float on a precision-32 engine, double
 * on a precision-64 engine).  Same conventions as uhc_b200.h: 0 on success, < 0 on error with uhc_last_error() set.
 */
#ifndef UHC_MOTION_H
#define UHC_MOTION_H
#include "uhc_b200.h"
#ifdef __cplusplus
extern "C" {
#endif

/* C clips of clip_len[c] >= 2 frames.  pose_host = concatenated [sum(len)][pose_dim] axis-angle rows: pose_dim 72 (SMPL, 24 joints) or 156
 * (SMPL-H: the first 22 joints are kept, the hands set to zero, as smplh_to_smpl does); trans_host = [sum(len)][3] root translations or NULL
 * (every clip at (0, 0, 0.91437225)); shape_host = [C][17] (beta16, gender); clip_model_host = [C] body-shape variant of every clip or NULL
 * (variant 0).  Each clip's records use its variant's bone offsets, centres of mass and root offset.
 * Side effects are those of uhc_load_clips followed by uhc_set_clip_models: every env record is invalidated, the clip sampling weights
 * return to their default, the clip models are set.  A rejected call (bad argument, clip_model out of range, a non-finite pose / trans /
 * shape value) returns < 0 and leaves the previous table in place. */
int uhc_load_clips_smpl(UhcEngine *e, int nclips, const int *clip_len, int pose_dim, const double *pose_host, const double *trans_host,
                        const double *shape_host, const int *clip_model_host);

/* rows [frame0, frame0 + nframes) of the engine's clip table (frames of all clips, concatenated in clip order) -> out_host
 * [nframes][UHC_EX_SIZE] doubles: the ground truth as the kernels read it. */
int uhc_get_clip_frames(UhcEngine *e, int frame0, int nframes, double *out_host);

#ifdef __cplusplus
}
#endif
#endif
