"""Builds libnic.so (sm_100a) in-tree with nvcc.  `python -m neural_image_compression_v2_b200.build`.

nvcc cross-compiles without a GPU; the resulting .so is git-ignored but travels with the gpurun snapshot."""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libnic.so")
# (source, extra defines, object name)
UNITS = [("nic_api.cu", [], "nic_api.o"), ("nic_f32.cu", [], "nic_f32.o"), ("nic_optim.cu", [], "nic_optim.o"),
         ("nic_tc.cu", [], "nic_tc.o"), ("nic_gather.cu", [], "nic_gather.o"), ("nic_train_tc.cu", [], "nic_train_tc.o"),
         ("nic_data.cu", [], "nic_data.o"), ("nic_sample.cu", [], "nic_sample.o"), ("nic_lut.cu", [], "nic_lut.o"),
         ("nic_f32_mlp.cu", ["-DNIC_H=64", "-DNIC_PART=0"], "nic_f32_fwd64.o"),
         ("nic_f32_mlp.cu", ["-DNIC_H=64", "-DNIC_PART=1"], "nic_f32_bwd64.o"),
         ("nic_f32_mlp.cu", ["-DNIC_H=32", "-DNIC_PART=0"], "nic_f32_fwd32.o"),
         ("nic_f32_mlp.cu", ["-DNIC_H=32", "-DNIC_PART=1"], "nic_f32_bwd32.o")]
EXTRA = os.environ.get("NIC_EXTRA_NVCC_FLAGS", "").split()
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr"]


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "nic.h"))
    jobs = []
    for src, defs, obj in UNITS:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, obj)
        if force or _stale(o, [s] + headers):
            jobs.append((s, defs, o))

    def compile_one(job):
        s, defs, o = job
        r = subprocess.run([_nvcc()] + NVCC_FLAGS + EXTRA + defs + ["-c", s, "-o", o], capture_output=True, text=True)
        with open(o + ".log", "w") as f:
            f.write(r.stdout + r.stderr)
        return s, r

    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        for s, r in ex.map(compile_one, jobs):
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {s}:\n{r.stdout}\n{r.stderr}")
            if verbose:
                print(r.stderr)
    objs = [os.path.join(OBJ, u[2]) for u in UNITS]
    if force or jobs or _stale(LIB, objs):
        r = subprocess.run([_nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
