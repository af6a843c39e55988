"""Builds libuhc_b200.so (CUDA, sm_100a) in-tree.  nvcc cross-compiles without a GPU."""
import os
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libuhc_b200.so")
SRCS = ["step_kernel.cu", "nn_kernels.cu", "mlp_tcgen05.cu", "rollout.cu", "ppo_update.cu", "eval.cu"]
# compiled on their own without FMA contraction: the device motion library keeps the operation order of the host numpy code it restates
SRCS_NOFMA = ["motion_lib.cu"]
DEPS = ["sim_core.h", "env_step.h", "eval_internal.h", "eval_metrics.h", "clip_table.h", "motion_fk.h", "../../include/uhc_b200.h", "../../include/uhc_nn.h",
        "../../include/uhc_rollout.h", "../../include/uhc_ppo.h", "../../include/uhc_eval.h", "../../include/uhc_motion.h"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--use_fast_math=false",
              "-Xcompiler", "-fPIC", "-shared", "-Xptxas", "-v", "--expt-relaxed-constexpr"]


def build(force=False, verbose=False):
    csrc = os.path.join(HERE, "csrc")
    srcs = [os.path.join(csrc, s) for s in SRCS]
    nofma = [os.path.join(csrc, s) for s in SRCS_NOFMA]
    deps = srcs + nofma + [os.path.join(csrc, d) for d in DEPS] + [os.path.abspath(__file__)]
    if not force and os.path.exists(SO) and os.path.getmtime(SO) >= max(os.path.getmtime(d) for d in deps if os.path.exists(d)):
        return SO
    flags = [f for f in NVCC_FLAGS if f != "--use_fast_math=false"] + os.environ.get("UHC_NVCC_EXTRA", "").split()
    with tempfile.TemporaryDirectory() as tmp:
        objs = [os.path.join(tmp, os.path.basename(s) + ".o") for s in nofma]
        cmds = [["nvcc"] + [f for f in flags if f != "-shared"] + ["-fmad=false", "-c", "-o", o, s] for s, o in zip(nofma, objs)]
        cmds.append(["nvcc"] + flags + ["-o", SO] + srcs + objs + ["-ldl"])
        for cmd in cmds:
            r = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or r.returncode:
                print(r.stdout[-6000:], r.stderr[-12000:])
            if r.returncode:
                raise RuntimeError("nvcc failed")
    return SO


if __name__ == "__main__":
    build(force=True, verbose=True)
