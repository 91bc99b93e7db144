"""In-tree build of libdkb.so for sm_100a (explicit nvcc; the .so travels with gpurun).

The scan kernel's instantiations are compiled one probe stride per translation unit
(csrc/dkb_scan_inst.cu with -DDKB_INST_D=1|2|4|8|16), in parallel with the rest of the library
(csrc/dkb_api.cu, csrc/dkb_host.cpp); objects go to build/ and are linked into libdkb.so."""
import hashlib
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
HEADERS = [os.path.join(CSRC, f) for f in ("dkb_device.cuh", "dkb_scan.cuh", "dkb_build.cuh", "dkb_pack.cuh",
                                              "dkb_regions.cuh")] + [
    os.path.join(_HERE, "..", "include", "dkb.h")]
STRIDES = (1, 2, 4, 8, 16)
OUT = os.path.join(_HERE, "libdkb.so")
OBJ_DIR = os.path.join(_HERE, "..", "build", "dkb")
NVCC_FLAGS = ["-Xcompiler", "-fPIC", "-std=c++17", "-O3", "-lineinfo",
              "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "g++", "-Xcompiler", "-pthread"]


def units(extra=()):
    """(object name, source, flags) of every translation unit."""
    u = [("dkb_api.o", os.path.join(CSRC, "dkb_api.cu"), []),
         ("dkb_host.o", os.path.join(CSRC, "dkb_host.cpp"), [])]
    u += [(f"dkb_scan_d{d}.o", os.path.join(CSRC, "dkb_scan_inst.cu"), [f"-DDKB_INST_D={d}"]) for d in STRIDES]
    return [(o, s, f + list(extra)) for o, s, f in u]


def _stamp(src, flags):
    h = hashlib.sha1()
    for p in [src] + HEADERS:
        with open(p, "rb") as f:
            h.update(f.read())
    h.update(" ".join(flags).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False, out: str = OUT, extra=(), obj_dir: str = OBJ_DIR) -> str:
    nvcc = os.environ.get("NVCC", "nvcc")
    # fast path (a GPU box receives the built library but not build/): up to date by mtime
    srcs = {s for _, s, _ in units(extra)} | set(HEADERS)
    if not force and os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(p) for p in srcs):
        return out
    os.makedirs(obj_dir, exist_ok=True)
    todo, objs = [], []
    for obj, src, flags in units(extra):
        path = os.path.join(obj_dir, obj)
        objs.append(path)
        stamp = _stamp(src, NVCC_FLAGS + flags)
        try:
            with open(path + ".stamp") as f:
                fresh = f.read() == stamp and os.path.exists(path)
        except OSError:
            fresh = False
        if force or not fresh:
            todo.append((path, src, flags, stamp))
    if not todo and os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(o) for o in objs):
        return out

    def compile_one(job):
        path, src, flags, stamp = job
        cmd = [nvcc] + NVCC_FLAGS + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", path, src]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"{' '.join(cmd)}\n{r.stdout}\n{r.stderr}")
        with open(path + ".stamp", "w") as f:
            f.write(stamp)
        return r.stderr

    with ThreadPoolExecutor(max_workers=min(len(todo), os.cpu_count() or 4) or 1) as ex:
        for log in ex.map(compile_one, todo):
            if verbose and log:
                print(log)
    subprocess.check_call([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "g++",
                           "-Xcompiler", "-pthread", "-o", out] + objs + ["-ldl"])
    return out


if __name__ == "__main__":
    print(build(force=True, verbose=True))
