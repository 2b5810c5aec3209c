"""Builds tacorl_b200/lib/libtacorl_b200.so with nvcc for sm_100a (no torch dependency)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
LIBDIR = os.path.join(os.path.dirname(HERE), "lib")
SOURCES = ["api.cu", "gemm_f32.cu", "gemm_tc.cu", "conv_tc.cu", "conv_f32.cu", "encoder.cu", "rnn.cu", "losses.cu", "optim.cu", "cql.cu", "transformer.cu", "mlp_chain.cu", "data_pipeline.cu", "dp_nccl.cu", "gripper.cu", "replay.cu", "rollout.cu", "plan_search.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-cudart", "static"]


def build(verbose=False, force=False):
    os.makedirs(LIBDIR, exist_ok=True)
    out = os.path.join(LIBDIR, "libtacorl_b200.so")
    srcs = [os.path.join(HERE, s) for s in SOURCES if os.path.exists(os.path.join(HERE, s))]
    deps = srcs + [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(os.path.dirname(os.path.dirname(HERE)), "include", "tacorl_b200.h"))
    if not force and os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(d) for d in deps):
        return out
    objs = []
    procs = []
    for s in srcs:
        o = os.path.join(LIBDIR, os.path.basename(s)[:-3] + ".o")
        cmd = ["nvcc"] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    failed = False
    for s, p in procs:
        log, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {os.path.basename(s)}\n{log}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = ["nvcc", "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out] + objs + ["-ldl"]
    subprocess.check_call(cmd)
    return out


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force=True))
