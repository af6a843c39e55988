// clip_table.h -- what the device motion library (motion_lib.cu) needs from the engine (step_kernel.cu); not part of the C ABI.
#pragma once
#include "../../include/uhc_b200.h"

// host fp64 copies of the kinematic tables of the engine's body-shape variants
struct EngineKin {
    const double *off_ipos;   // [nshape][24][6]: body offset, centre of mass (UhcModelHost.body_f columns 0..5)
    const int *parent, *ee;   // [24], [5]
    int nshape, precision, device;
};
int uhc_engine_kin(const UhcEngine *e, EngineKin *out);

// installs a clip table whose frames ([sum(clip_len)][UHC_EX_SIZE] of the engine's precision) and shapes ([nclips][17], same precision)
// already sit on the device; the engine owns both buffers from here on.  Everything uhc_load_clips does besides building the table: the
// previous table is freed, every env record invalidated, the clip weights reset to the sample_keys rule and the clip models cleared.
int uhc_engine_install_clips(UhcEngine *e, int nclips, const int *clip_len, void *expert_dev, void *shape_dev);

// the message uhc_last_error() returns
void uhc_engine_set_error(const char *msg);
