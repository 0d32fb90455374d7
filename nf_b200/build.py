"""Build libnisb200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libnisb200.so")
SOURCES = ["flow_desc.cu", "flow_fwd.cu", "flow_tiled.cu", "flow_tc_h.cu", "flow_wide.cu", "flow_bwd.cu", "flow_bwd_tc.cu", "flow_bwd_wide.cu", "rambo.cu", "reduce.cu", "probe_tc.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "nis_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def _compile_one(args):
    src, obj, verbose = args
    cmd = [_nvcc()] + NVCC_FLAGS[:-3] + ["-Xcompiler", "-fPIC"] + (["-Xptxas", "-v"] if verbose else []) + \
          ["-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    return src, r.returncode, r.stdout + r.stderr


def build(force=False, verbose=False):
    """Compile every .cu under nf_b200/csrc (one object per source, in parallel; objects are reused while the
    source and every header are older) and link nf_b200/libnisb200.so.  Returns the library path."""
    from concurrent.futures import ThreadPoolExecutor
    objdir = os.path.join(HERE, "csrc", "_obj")
    os.makedirs(objdir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))] + \
              [os.path.join(HERE, "..", "include", "nis_b200.h"), os.path.abspath(__file__)]
    hdr_t = max(os.path.getmtime(h) for h in headers)
    jobs, objs = [], []
    for sname in SOURCES:
        src = os.path.join(CSRC, sname)
        obj = os.path.join(objdir, sname[:-3] + ".o")
        objs.append(obj)
        if force or verbose or not os.path.exists(obj) or os.path.getmtime(obj) < max(hdr_t, os.path.getmtime(src)):
            jobs.append((src, obj, verbose))
    log = ""
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        for src, rc, out in ex.map(_compile_one, jobs):
            if rc != 0:
                raise RuntimeError("nvcc failed on %s:\n%s" % (src, out))
            log += out
    r = subprocess.run([_nvcc(), "-shared", "-Xcompiler", "-fPIC"] + NVCC_FLAGS[:2] + objs + ["-o", LIB + ".tmp"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    os.replace(LIB + ".tmp", LIB)
    if verbose:
        print(log)
    return LIB


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
