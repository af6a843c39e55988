// eval_internal.h -- what the evaluation loop (eval.cu) needs from the engine (step_kernel.cu); not part of the C ABI.
#pragma once
#include <cuda_runtime.h>
#include "../../include/uhc_b200.h"

namespace uhc { struct EvalView; }

// the engine's device clip table: frames [total][UHC_EX_SIZE] of float (precision 32) or double (64), clip_adr [C+1] on the device,
// clip_len [C] on the host
struct EngineTable {
    const void *expert;
    const int *clip_adr;
    const int *clip_len;
    int precision, num_clips, trail_steps, device;
};

// one control step of every env slot in evaluation mode (k_env_step<Real, EPB, true>); stream-ordered, no host synchronisation
int uhc_env_step_eval(UhcEngine *e, const float *actions_dev, float *obs_dev, float *reward_dev, int *fail_dev, int *end_dev, const uhc::EvalView &xv,
                      cudaStream_t st);
int uhc_engine_expert_table(const UhcEngine *e, EngineTable *out);
// uhc_env_reset (host arguments, start from the clip's frames, observations into obs_dev) with the engine's auto_reset cleared for the
// launch: no reactive standing-neutral starts, exactly the reset the evaluation-mode step kernel runs for the clips it takes from the queue
int uhc_env_reset_eval(UhcEngine *e, int n, const int *env_ids_host, const int *clip_host, const int *start_host, const int *len_host, float *obs_dev,
                       cudaStream_t st);
