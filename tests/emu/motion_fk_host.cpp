// host build of the expert-table math (uhc_b200/csrc/motion_fk.h) for the CPU test: the same per-frame code the CUDA kernel of
// uhc_load_clips_smpl runs
#include <stddef.h>
#include "../../uhc_b200/csrc/motion_fk.h"

extern "C" void motion_fk_host(const double *pose, int T, int pose_dim, const double *trans, const double *off_ipos, const int *parent, const int *ee,
                               double *out) {
    const uhc_motion::Kin k{off_ipos, parent, ee};
    for (int t = 0; t < T; t++) uhc_motion::expert_frame<double>(pose, pose_dim, trans, t, k, out + (size_t)uhc_motion::REC * t);
}

extern "C" void motion_smpl_joint(int *out) { for (int b = 0; b < uhc_motion::NB; b++) out[b] = uhc_motion::smpl_joint(b); }
