"""Build tests/emu/_build/ptr/libpelestencil_emu_ptr.so: the emulated library of build_emu.py (same sources, same flags) with
tests/emu/cuemu_pointer.h force-included and cuemu_pointer.cpp linked in, so cudaPointerGetAttributes tells the library's
and the tests' device blocks from host memory (TEST INFRASTRUCTURE; see cuemu_pointer.h).  asan=True builds the same with
AddressSanitizer into _build/ptr_asan."""
import os
import subprocess

import build_emu

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(HERE, "cuemu_pointer.h")
EXTRA = os.path.join(HERE, "cuemu_pointer.cpp")


def lib_path(asan: bool = False) -> str:
    return os.path.join(build_emu.OUT, "ptr_asan" if asan else "ptr", "libpelestencil_emu_ptr.so")


def _needs_build(lib: str) -> bool:
    if not os.path.exists(lib):
        return True
    t = os.path.getmtime(lib)
    deps = [s for s in build_emu.SOURCES] + [os.path.join(build_emu.CSRC, f) for f in os.listdir(build_emu.CSRC)]
    deps += [HEADER, EXTRA, os.path.abspath(__file__), os.path.join(HERE, "cuda_runtime.h"),
             os.path.join(build_emu.ROOT, "include", "pele_stencil_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(asan: bool = False, force: bool = False) -> str:
    lib = lib_path(asan)
    if not force and not _needs_build(lib):
        return lib
    out = os.path.dirname(lib)
    os.makedirs(out, exist_ok=True)
    san = ["-fsanitize=address", "-fno-omit-frame-pointer"] if asan else []
    import fcntl
    with open(os.path.join(out, ".build.lock"), "w") as lk:          # pytest-xdist workers share this directory
        fcntl.flock(lk, fcntl.LOCK_EX)
        if not force and not _needs_build(lib):
            return lib
        procs = []
        for s in build_emu.SOURCES + [EXTRA]:
            o = os.path.join(out, os.path.basename(s).rsplit(".", 1)[0] + ".o")
            # the kernel sources see the tracked allocator; cuemu.cpp and cuemu_pointer.cpp keep the plain one underneath
            inc = ["-include", HEADER] if os.path.dirname(os.path.abspath(s)) == build_emu.CSRC else []
            cmd = ["g++", *build_emu.FLAGS, *san, *inc, "-x", "c++", "-c", s, "-o", o]
            procs.append((s, o, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        for s, o, p in procs:
            txt, _ = p.communicate()
            if p.returncode != 0:
                raise RuntimeError("g++ failed on %s:\n%s" % (s, txt))
        subprocess.check_call(["g++", "-shared", *san, "-o", lib + ".tmp"] + [o for _, o, _ in procs])
        os.replace(lib + ".tmp", lib)
    return lib


if __name__ == "__main__":
    print(build(force=True))
