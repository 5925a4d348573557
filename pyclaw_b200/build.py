"""Builds the CUDA library in-tree with nvcc for sm_100a.

    python -m pyclaw_b200.build [--force] [-v] [--fma | --all]
    python -m pyclaw_b200.build --user-rp my_rp.cuh [--name mine] [--fma] [--ndims 3]   (plugin seam, see below)

Two builds of the same sources:
  libclawb200.so      -fmad=false : strict IEEE, bit-for-bit agreement with the reference's
                      Fortran (compiled without FMA contraction) -- the default, and the one every
                      parity test runs;
  libclawb200_fma.so  -fmad=true  : nvcc may contract a*b+c into one DFMA (fewer FP64-pipe
                      instructions); results differ from the strict build at round-off level
                      (measured in profiles/README.md), selected with solver.arithmetic = 'fma'.
-lineinfo keeps the ncu source page usable.

Riemann-solver plugin seam: `--user-rp header.cuh` compiles a user-supplied solver (a header with
`template <int IXY> struct RpUser`, see examples/user_rp/rp_kpp.cuh, and/or the 3-D
`template <int IXYZ> struct RpUser3`, see examples/user_rp/rp_acoustics3d_user.cuh, selected with
`--ndims 3` or `--ndims 1,2,3`) into libclawb200_user_<name>.so -- the reference does the same at link time with RP_SOURCE in each
application's Makefile (Makefile.rules:1-26).  pyclaw.riemann.from_header() builds and binds it.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libclawb200.so")
LIB_FMA = os.path.join(CSRC, "libclawb200_fma.so")
# translation units (compiled in parallel, linked into one shared library) and what each includes
_COMMON = ["arith.cuh", "rp.cuh", "classic.cuh", "launch.cuh", os.path.join("..", "..", "include", "clawb200.h")]
UNITS = {
    "clawb200.cu": _COMMON,
    "sweep_euler_x.cu": _COMMON,
    "sweep_euler_y.cu": _COMMON,
    "sweep_sphere.cu": _COMMON,
    "sweep_misc.cu": _COMMON,
    "sweep_fused.cu": _COMMON + ["fused.cuh"],
    "step1.cu": _COMMON,
    "step3.cu": _COMMON + ["step3.cuh"],          # 3-D steps (step3.cuh): vc-acoustics
    "step3_euler.cu": _COMMON + ["step3.cuh"],    # ... 3-D Euler
    "step3_misc.cu": _COMMON + ["step3.cuh"],     # ... 3-D advection, 3-D f-wave transport
    "rp_point.cu": _COMMON + ["rp_point.cuh"],
    "sharpclaw.cu": _COMMON + ["sharpclaw.cuh"],
    "sharpclaw3.cu": _COMMON + ["sharpclaw.cuh", "sharpclaw3.cuh"],        # 3-D SharpClaw stage: vc-acoustics
    "sharpclaw3_euler.cu": _COMMON + ["sharpclaw.cuh", "sharpclaw3.cuh"],  # ... 3-D Euler
    "sharpclaw3_misc.cu": _COMMON + ["sharpclaw.cuh", "sharpclaw3.cuh"],   # ... 3-D advection, 3-D f-wave transport
    "sweep_user.cu": _COMMON + ["rp_point.cuh", "sharpclaw.cuh", "sharpclaw3.cuh", "step3.cuh"],   # the user-supplied Riemann solver (a stub without one)
}
SOURCES = list(UNITS)
HEADERS = sorted({h for hs in UNITS.values() for h in hs})

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
]


def _stale(lib):
    if not os.path.exists(lib):
        return True
    t = os.path.getmtime(lib)
    for f in SOURCES + HEADERS:
        if os.path.getmtime(os.path.join(CSRC, f)) > t:
            return True
    return False


def _obj_stale(obj, src):
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in [src] + UNITS[src])


def build(force=False, verbose=False, fma=False, jobs=None):
    """Compile the translation units (object files under csrc/_obj/, only the stale ones unless
    `force`) with up to `jobs` nvcc processes, then link the shared library."""
    from concurrent.futures import ThreadPoolExecutor
    lib = LIB_FMA if fma else LIB
    if not force and not _stale(lib):
        return lib
    nvcc = os.environ.get("NVCC", "nvcc")
    flags = NVCC_FLAGS + (["-fmad=true", "-DCLAWB200_FMA=1"] if fma else ["-fmad=false"])
    if verbose:
        flags = flags + ["-Xptxas", "-v"]
    objdir = os.path.join(CSRC, "_obj", "fma" if fma else "strict")
    os.makedirs(objdir, exist_ok=True)
    objs, todo = [], []
    for src in SOURCES:
        obj = os.path.join(objdir, src[:-3] + ".o")
        objs.append(obj)
        if force or _obj_stale(obj, src):
            todo.append((src, obj))

    def compile_one(job):
        src, obj = job
        r = subprocess.run([nvcc] + flags + ["-c", "-o", obj, src], cwd=CSRC, capture_output=True, text=True)
        return src, r
    jobs = jobs or min(len(todo), os.cpu_count() or 1) or 1
    failed = None
    with ThreadPoolExecutor(max_workers=jobs) as ex:
        for src, r in ex.map(compile_one, todo):
            if verbose or r.returncode != 0:
                sys.stderr.write("==== %s ====\n%s%s" % (src, r.stdout, r.stderr))
            if r.returncode != 0:
                failed = src
    if failed:
        raise subprocess.CalledProcessError(1, "nvcc -c " + failed)
    # link under a temporary name and rename: a reader (a gpurun snapshot, a running process that
    # dlopens the library) sees either the old or the new file, never a half-written one
    subprocess.check_call([nvcc, "-shared", "-o", lib + ".tmp"] + objs, cwd=CSRC)
    os.replace(lib + ".tmp", lib)
    return lib


def user_lib_path(name, fma=False):
    return os.path.join(CSRC, "libclawb200_user_%s%s.so" % (name, "_fma" if fma else ""))


def user_flags(ndims):
    """The defines that tell csrc/sweep_user.cu which structs the header has: RpUser (1-D / 2-D)
    unless `ndims` lacks 1 and 2, RpUser3 when it contains 3."""
    flags = []
    if 3 in ndims:
        flags.append("-DCLAWB200_USER_RP3")
    if not set(ndims) & {1, 2}:
        flags.append("-DCLAWB200_USER_NO_RP")
    return flags


def build_user(header, name=None, fma=False, force=False, verbose=False, ndims=(1, 2)):
    """A variant of the library with a user-supplied Riemann solver (csrc/sweep_user.cu): the
    header defines `template <int IXY> struct RpUser` (ndims 1, 2) and / or `template <int IXYZ>
    struct RpUser3` (ndims 3) with the interfaces of the solvers in rp.cuh.  Only sweep_user.cu is
    compiled; every other object comes from the base build.
    Returns the path of libclawb200_user_<name>[_fma].so."""
    header = os.path.abspath(header)
    if not os.path.exists(header):
        raise FileNotFoundError(header)
    name = name or os.path.splitext(os.path.basename(header))[0]
    build(fma=fma)  # base objects
    lib = user_lib_path(name, fma)
    deps = [header] + [os.path.join(CSRC, f) for f in ["sweep_user.cu"] + UNITS["sweep_user.cu"]]
    base_lib = LIB_FMA if fma else LIB
    if not force and os.path.exists(lib) and all(os.path.getmtime(d) <= os.path.getmtime(lib) for d in deps + [base_lib]):
        return lib
    nvcc = os.environ.get("NVCC", "nvcc")
    flags = NVCC_FLAGS + (["-fmad=true", "-DCLAWB200_FMA=1"] if fma else ["-fmad=false"])
    objdir = os.path.join(CSRC, "_obj", "user_%s%s" % (name, "_fma" if fma else ""))
    os.makedirs(objdir, exist_ok=True)
    obj = os.path.join(objdir, "sweep_user.o")
    cmd = [nvcc] + flags + (["-Xptxas", "-v"] if verbose else []) + \
        ['-DCLAWB200_USER_RP_HEADER="%s"' % header] + user_flags(ndims) + ["-c", "-o", obj, "sweep_user.cu"]
    subprocess.check_call(cmd, cwd=CSRC)
    base = os.path.join(CSRC, "_obj", "fma" if fma else "strict")
    objs = [obj] + [os.path.join(base, s[:-3] + ".o") for s in SOURCES if s != "sweep_user.cu"]
    subprocess.check_call([nvcc, "-shared", "-o", lib + ".tmp"] + objs, cwd=CSRC)
    os.replace(lib + ".tmp", lib)
    return lib


def build_all(force=False):
    """Both builds, side by side (two nvcc processes)."""
    import threading
    out = {}
    ts = [threading.Thread(target=lambda f=f: out.__setitem__(f, build(force=force, fma=f))) for f in (False, True)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    return out[False], out[True]


if __name__ == "__main__":
    if "--user-rp" in sys.argv:
        hdr = sys.argv[sys.argv.index("--user-rp") + 1]
        nm = sys.argv[sys.argv.index("--name") + 1] if "--name" in sys.argv else None
        nd = tuple(int(d) for d in sys.argv[sys.argv.index("--ndims") + 1].split(",")) if "--ndims" in sys.argv else (1, 2)
        print(build_user(hdr, nm, fma="--fma" in sys.argv, force="--force" in sys.argv, verbose="-v" in sys.argv,
                         ndims=nd))
    elif "--all" in sys.argv:
        print(*build_all(force="--force" in sys.argv))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, fma="--fma" in sys.argv))
