"""TEST INFRASTRUCTURE: libfplgpu and the drop-in binary without a GPU.

`build_library()` builds every .cu of fastplong_b200/csrc — fpl_api.cu with the C ABI, run_batch and the accumulators, fpl_jit.cu
with its code generator, all kernels — for the HOST: the source text is preprocessed (`mad.lo.u32` inline PTX rewritten as C, the
small PTX wrappers cut out in favour of host forms, `extern __shared__` bound to the emulator's buffer, `kernel<<<grid, block,
smem, stream>>>(args)` turned into a call of the SIMT emulator) and compiled with g++ against tests/simt/fake/ — a host-memory
<cuda_runtime.h> (device memory is host memory, streams are synchronous, events are timestamps), host stand-ins for the three
cub primitives, and an NVRTC + driver shim (tests/simt/emu_core.cpp) under which fpl_jit.cu "compiles" the kernel source it
generates with g++ and "loads the cubin" with dlopen.  Kernels run under tests/simt/emu_cuda.h: one OS thread, every CUDA thread
of a block a fiber, warp / block collectives with their real semantics, cp.async completing at the latest legal moment, mbarrier
phases with transaction counts.  The result, libfplgpu_emu.so, exports include/fplgpu.h like libfplgpu.so does.

`build_binary()` links host/seprocessor_gpu.cpp, unchanged, with the reference's objects against it: the drop-in CLI.
`EmuEngine` is binding.Engine on the emulated library (what tests/test_simt_kernels.py and tools/fuzz_emulated_vs_oracle.py
use); `FPL_EMULATE=1` (tests/conftest.py) runs the `-m gpu` test files on the same build.

Not modelled: timing, caches, bank conflicts, memory ordering between warps, the NCCL merge; cub's own kernels are stood in for.
Nothing here is shipped or reachable from the product path.
"""
import ctypes as C
import hashlib
import os
import re
import subprocess

from device_helpers import CSRC, ROOT, _asm_to_c, _match_brace

SIMT = os.path.join(ROOT, "tests", "simt")
PTX_WRAPPERS = ("prmt", "cp_async16", "cp_async4", "cp_async_commit", "cp_async_wait", "lds128", "lds32", "mbar_init", "mbar_expect_tx",
                "mbar_wait", "bulk_g2s", "red_shared_add_imm")


def _drop_function(text, name):
    m = re.search(r"^(?:template\s*<[^>\n]*>\s*\n)?[A-Za-z_][^\n;{}()]*\b" + name + r"\s*\([^;{}]*\)\s*\{", text, re.M)
    if not m:
        raise KeyError(name)
    end = _match_brace(text, m.end() - 1)
    return text[:m.start()] + text[end + 1:]


def _split_top(s):
    out, depth, cur = [], 0, ""
    for ch in s:
        if ch in "([{":
            depth += 1
        elif ch in ")]}":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur.strip())
            cur = ""
        else:
            cur += ch
    out.append(cur.strip())
    return out


def _rewrite_launches(text):
    out, i = "", 0
    while True:
        j = text.find("<<<", i)
        if j < 0:
            return out + text[i:]
        k = text.index(">>>", j)
        # kernel name (with template arguments) in front of <<<
        m = re.search(r"([A-Za-z_]\w*(?:<[^<>;]*>)?)\s*$", text[:j])
        cfg = _split_top(text[j + 3:k])
        p = text.index("(", k)
        q = p
        depth = 0
        while True:
            depth += text[q] == "("
            depth -= text[q] == ")"
            if depth == 0:
                break
            q += 1
        smem = cfg[2] if len(cfg) > 2 else "0"
        out += text[i:m.start()] + f"EMU_LAUNCH(({cfg[0]}), ({cfg[1]}), ({smem}), {m.group(1)}{text[p:q + 1]})"
        i = q + 1


# ---- the build ----
LIB_SOURCES = ("fpl_api.cu", "fpl_trim.cu", "fpl_scan.cu", "fpl_scan_fast.cu", "fpl_stats.cu", "fpl_jit.cu", "fpl_ingest.cu", "fpl_ext.cu",
               "fpl_eval.cu", "fpl_emit.cu")


def _lib_text(fn, text=None):
    text = open(os.path.join(CSRC, fn)).read() if text is None else text
    drops = {"fpl_device.cuh": ("red_shared_add", "shared_addr"), "fpl_stats.cu": PTX_WRAPPERS}.get(fn, ())
    for name in drops:
        text = _drop_function(text, name)
    text = re.sub(r"extern\s+__shared__\s+(?:__align__\(\d+\)\s+)?(\w+)\s+(\w+)\[\];", r"\1* \2 = (\1*)emu::dynamic_smem;", text)
    text = re.sub(r'asm\s+volatile\s*\(\s*"fence[^"]*"[^;]*;', ";", text)
    text = text.replace('dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL)', "dlopen(EMU_LIB_PATH, RTLD_NOW)")
    return _rewrite_launches(_asm_to_c(text))


_emu_lib_path = None


def build_library(override=None):
    """-> path of libfplgpu_emu.so (built once per source state into /tmp).  override: {file name: source text} replacing files of
    fastplong_b200/csrc (tools/mutate_kernels.py builds mutants this way; such builds are not remembered as THE library)."""
    global _emu_lib_path
    if _emu_lib_path and not override:
        return _emu_lib_path
    files = {}
    for fn in sorted(os.listdir(CSRC)):
        if fn.endswith((".cu", ".cuh", ".h")):
            files[fn] = _lib_text(fn, (override or {}).get(fn))
    extra = ""
    for root, _, names in os.walk(SIMT):
        for nm in sorted(names):
            extra += open(os.path.join(root, nm)).read()
    san = os.environ.get("FPL_EMU_SANITIZE", "")          # e.g. "undefined": the kernels and fpl_api.cu's host code under UBSan
    tag = hashlib.md5(("".join(files[k] for k in sorted(files)) + extra + san).encode()).hexdigest()[:12]
    out = f"/tmp/fpl_emu_lib_{tag}"
    so = os.path.join(out, "libfplgpu_emu.so")
    if not os.path.exists(so):
        os.makedirs(out, exist_ok=True)
        for fn, text in files.items():
            open(os.path.join(out, fn[:-3] + ".cpp" if fn.endswith(".cu") else fn), "w").write(text)
        defs = [f'-DEMU_LIB_PATH="{so}"', f'-DEMU_LIB_DIR="{out}"', f'-DEMU_SIMT_DIR="{SIMT}"', f'-DEMU_BUILD_TAG="{tag}"']
        inc = ["-I", out, "-I", os.path.join(SIMT, "fake"), "-I", SIMT, "-I", os.path.join(ROOT, "include")]
        objs = []
        jobs = []
        for src in [os.path.join(out, fn[:-3] + ".cpp") for fn in LIB_SOURCES] + [os.path.join(SIMT, "emu_core.cpp")]:
            obj = os.path.join(out, os.path.basename(src)[:-4] + ".o")
            objs.append(obj)
            sflags = [f"-fsanitize={san}", "-fno-omit-frame-pointer"] if san else []        # reports go to stderr, the run goes on
            jobs.append(subprocess.Popen(["g++", "-std=c++17", "-O1", "-g", "-fPIC", "-w", "-c", *sflags, *defs, *inc, "-o", obj, src],
                                         stderr=subprocess.PIPE, text=True))
        for j in jobs:
            err = j.communicate()[1]
            if j.returncode != 0:
                raise RuntimeError("emulated build failed:\n" + err[:6000])
        subprocess.check_call(["g++", "-shared", *([f"-fsanitize={san}"] if san else []), "-o", so + ".tmp", *objs, "-ldl", "-lpthread"])
        os.replace(so + ".tmp", so)
    if not override:
        _emu_lib_path = so
    return so


_emu_bin_path = None


def _reference_src():
    """The reference's source directory, whose headers seprocessor_gpu.cpp includes: oracle/Makefile's REF (which the
    environment may override), so that the emulated build and the Makefiles read the same sources."""
    r = subprocess.run(["make", "-s", "--no-print-directory", "-C", os.path.join(ROOT, "oracle"), "print-ref"],
                       capture_output=True, text=True)
    return os.path.join(r.stdout.strip(), "src") if r.returncode == 0 and r.stdout.strip() else None


REF_SRC = _reference_src()


def build_binary():
    """-> path of fastplong_gpu_emu: host/seprocessor_gpu.cpp (unchanged) + the reference's unmodified objects (oracle/_ref/obj, as
    fastplong_b200/host/Makefile links them) + the emulated library.  The drop-in CLI without a GPU."""
    global _emu_bin_path
    if _emu_bin_path:
        return _emu_bin_path
    lib = build_library()
    out = os.path.dirname(lib)
    exe = os.path.join(out, "fastplong_gpu_emu")
    host = os.path.join(ROOT, "fastplong_b200", "host", "seprocessor_gpu.cpp")
    objdir = os.path.join(ROOT, "oracle", "_ref", "obj")
    stamp = os.path.join(out, "host.md5")
    tag = hashlib.md5(open(host, "rb").read()).hexdigest()
    if not os.path.exists(exe) or not os.path.exists(stamp) or open(stamp).read() != tag:
        if not os.path.exists(os.path.join(objdir, "main.o")):
            raise RuntimeError("oracle/_ref/obj is not built (make -C oracle)")
        obj = os.path.join(out, "seprocessor_gpu.o")
        san = os.environ.get("FPL_EMU_SANITIZE", "")
        sflags = [f"-fsanitize={san}", "-fno-omit-frame-pointer", "-g"] if san else []
        subprocess.check_call(["g++", "-std=c++14", "-pthread", "-O2", "-w", *sflags, "-I", os.path.join(SIMT, "fake"), "-I", os.path.join(ROOT, "oracle", "shim"),
                               "-I", REF_SRC, "-I", os.path.join(ROOT, "include"), "-c", host, "-o", obj])
        refobj = sorted(os.path.join(objdir, f) for f in os.listdir(objdir)
                        if f.endswith(".o") and f not in ("seprocessor.o", "seprocessor_gpu.o"))
        subprocess.check_call(["g++", "-pthread", *sflags[:1], "-o", exe, obj, *refobj, lib, "-lz", "-ldl", f"-Wl,-rpath,{out}"])
        open(stamp, "w").write(tag)
    _emu_bin_path = exe
    return exe


# ---- binding.Engine on the emulated library ----
def emulated_library():
    """ctypes handle of the emulated library (emulator switches: emu_set_cp_async_lazy, emu_collectives, emu_blocks)"""
    lib = C.CDLL(build_library())
    lib.emu_set_cp_async_lazy.argtypes = [C.c_int]
    lib.emu_collectives.restype = lib.emu_blocks.restype = C.c_longlong
    return lib


class _Bound:
    """binding's module state pointed at the emulated library for the duration of a `with` block"""

    def __enter__(self):
        from fastplong_b200 import binding
        self.binding, self.saved = binding, (binding.LIB_PATH, binding._lib)
        path = build_library()
        binding.LIB_PATH, binding._lib = path, _Bound.libs.get(path)
        _Bound.libs[path] = binding.load_library()
        return binding

    def __exit__(self, *exc):
        self.binding.LIB_PATH, self.binding._lib = self.saved


_Bound.libs = {}      # path -> loaded handle (a mutant build is another path)


def EmuEngine(options, scan="jit"):
    """binding.Engine(options) on the emulated library.  scan: which whole-read scan kernel fpl_create sets up — "jit": the default
    (k_scan_jit specialised through the NVRTC stand-in wherever the library specialises), "fast": FPL_NO_JIT=1 (the precompiled
    k_scan_fast), "generic": FPL_FORCE_GENERIC_SCAN=1 (k_scan)."""
    env = {"jit": {}, "fast": {"FPL_NO_JIT": "1"}, "generic": {"FPL_FORCE_GENERIC_SCAN": "1"}}[scan]
    saved = {k: os.environ.get(k) for k in ("FPL_NO_JIT", "FPL_FORCE_GENERIC_SCAN")}
    for k in saved:
        os.environ.pop(k, None)
    os.environ.update(env)
    try:
        with _Bound() as binding:
            return binding.Engine(options)
    finally:
        for k, v in saved.items():
            os.environ.pop(k, None)
            if v is not None:
                os.environ[k] = v


def eval_adapter_kmers(batch, side, shift_tail=1):
    """binding.eval_adapter_kmers (k_eval_kmers) on the emulated library"""
    with _Bound() as binding:
        return binding.eval_adapter_kmers(batch, side, shift_tail, 0)
