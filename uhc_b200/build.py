"""Builds libuhc_b200.so (CUDA, sm_100a) in-tree.  nvcc cross-compiles without a GPU."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libuhc_b200.so")
SRCS = ["step_kernel.cu", "nn_kernels.cu", "mlp_tcgen05.cu", "rollout.cu", "ppo_update.cu", "eval.cu"]
DEPS = ["sim_core.h", "env_step.h", "eval_internal.h", "eval_metrics.h", "../../include/uhc_b200.h", "../../include/uhc_nn.h", "../../include/uhc_rollout.h", "../../include/uhc_ppo.h", "../../include/uhc_eval.h"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--use_fast_math=false",
              "-Xcompiler", "-fPIC", "-shared", "-Xptxas", "-v", "--expt-relaxed-constexpr"]


def build(force=False, verbose=False):
    csrc = os.path.join(HERE, "csrc")
    srcs = [os.path.join(csrc, s) for s in SRCS]
    deps = srcs + [os.path.join(csrc, d) for d in DEPS] + [os.path.abspath(__file__)]
    if not force and os.path.exists(SO) and os.path.getmtime(SO) >= max(os.path.getmtime(d) for d in deps if os.path.exists(d)):
        return SO
    flags = [f for f in NVCC_FLAGS if f != "--use_fast_math=false"] + os.environ.get("UHC_NVCC_EXTRA", "").split()
    cmd = ["nvcc"] + flags + ["-o", SO] + srcs + ["-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode:
        print(r.stdout[-6000:], r.stderr[-12000:])
    if r.returncode:
        raise RuntimeError("nvcc failed")
    return SO


if __name__ == "__main__":
    build(force=True, verbose=True)
