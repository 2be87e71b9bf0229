"""CPU: the C-ABI library builds, loads, and exports exactly the symbols include/gnan_b200.h declares (no compute calls)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib_path():
    import importlib.util
    spec = importlib.util.spec_from_file_location("gnan_build", os.path.join(ROOT, "graph-neural-additive-networks---gnan_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


def header_functions():
    src = open(os.path.join(ROOT, "include", "gnan_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gnan_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported(lib_path):
    lib = ctypes.CDLL(lib_path)
    names = header_functions()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"{n} declared in gnan_b200.h but not exported"


def test_exports_are_exactly_the_header_functions(lib_path):
    """No C entry point outside the header: a caller cannot reach a function the ABI does not document. C++ helpers shared between
    the library's own files have mangled names (_Z...) and are not C entry points."""
    import subprocess
    out = subprocess.run(["nm", "-D", "--defined-only", lib_path], check=True, capture_output=True, text=True).stdout
    exported = sorted({f[-1] for f in (line.split() for line in out.splitlines()) if f and f[-1].startswith("gnan_")})
    assert exported == header_functions()


def test_python_binding_covers_the_version_102_header(lib_path):
    from gnan_b200 import _lib
    assert sorted(_lib.SIGNATURES) == header_functions()
    lib = _lib.load()
    assert lib.gnan_version() == 102
    assert lib.gnan_last_error() is not None


def test_argument_validation_of_the_surviving_entry_points_without_gpu(lib_path):
    """Validation happens before any CUDA call, so error codes can be checked on a CPU-only box."""
    from gnan_b200 import _lib
    lib = _lib.load()
    p = _lib.MlpParams(3, 24, 2, 3, None, None, None, None, None, None)   # H=24 unsupported, wo NULL
    rc = lib.gnan_mlp_fwd(None, 4, 3, ctypes.byref(p), 0.0, 0, None, 0, None, None, 0, None)
    assert rc == 1 and b"wo" in lib.gnan_last_error()
    rc = lib.gnan_aggregate_rows_fwd_ws(None, 4, 4, 16, None, 0, 5, 1, None, None, 1, None, None, 0, None, 0, None)
    assert rc == 1
    arr = (ctypes.c_int64 * 8)()
    buf = ctypes.addressof(arr)
    rc = lib.gnan_apsp_bfs_batched_ex(buf, buf, buf, buf, 1, 4, buf, None, None, 0, buf, None, None, None)   # order_ws NULL
    assert rc == 1 and b"order_ws" in lib.gnan_last_error()
    assert lib.gnan_mlp_workspace_bytes(0, ctypes.byref(p), 0, 0) == 0


C_CONSUMER = r"""
/* a plain C99 consumer of include/gnan_b200.h: the header must compile as C (no torch, no C++), the library must load with dlopen
   and report argument errors through int codes + gnan_last_error() */
#include <dlfcn.h>
#include <stdio.h>
#include <string.h>
#include "gnan_b200.h"

typedef int (*version_fn)(void);
typedef const char *(*error_fn)(void);
typedef int (*rscale_fn)(const int32_t *, int64_t, int32_t, float *, gnan_stream_t);
typedef size_t (*ws_fn)(int64_t, const gnan_mlp_params *, int, int);

int main(int argc, char **argv)
{
    void *h = dlopen(argv[1], RTLD_NOW);
    if (!h) { fprintf(stderr, "%s\n", dlerror()); return 2; }
    version_fn version; error_fn last_error; rscale_fn level_rscale; ws_fn mlp_ws;
    *(void **)(&version) = dlsym(h, "gnan_version");        /* the POSIX idiom for dlsym -> function pointer */
    *(void **)(&last_error) = dlsym(h, "gnan_last_error");
    *(void **)(&level_rscale) = dlsym(h, "gnan_level_rscale");
    *(void **)(&mlp_ws) = dlsym(h, "gnan_mlp_workspace_bytes");
    if (!version || !last_error || !level_rscale || !mlp_ws) return 3;
    gnan_mlp_params p;
    memset(&p, 0, sizeof p);
    p.G = 4; p.H = 64; p.C = 3; p.n_layers = 3;
    int rc = level_rscale(NULL, 4, 5, NULL, NULL);          /* NULL buffers: refused before any CUDA call */
    printf("%d %d %d %zu %s\n", version(), rc, (int)GNAN_PREC_TF32X3, mlp_ws(1000, &p, 1, GNAN_PREC_FP32), last_error());
    (void)argc;
    return 0;
}
"""


def test_c99_consumer_compiles_against_the_version_102_header_and_calls_the_library(lib_path, tmp_path):
    import subprocess
    src = tmp_path / "consumer.c"
    src.write_text(C_CONSUMER)
    exe = tmp_path / "consumer"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe), "-ldl"],
                   check=True, capture_output=True, text=True)
    out = subprocess.run([str(exe), lib_path], check=True, capture_output=True, text=True).stdout.split(None, 4)
    assert out[0] == "102" and int(out[1]) != 0 and out[2] == "1" and int(out[3]) >= 0 and "level_rscale" in out[4]
    # and as C++ (the reference-side binding may be either)
    subprocess.run(["g++", "-std=c++11", "-Wall", "-Werror", "-fsyntax-only", "-x", "c++", "-I", os.path.join(ROOT, "include"), str(src)],
                   check=True, capture_output=True, text=True)


def _header_prototypes():
    """{name: (return type, [parameter types])} parsed from include/gnan_b200.h (comments stripped, parameter names dropped)"""
    src = open(os.path.join(ROOT, "include", "gnan_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    protos = {}
    for ret, name, args in re.findall(r"^\s*((?:const\s+)?[A-Za-z_][A-Za-z0-9_]*(?:\s*\*)?)\s*(gnan_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", src, flags=re.M | re.S):
        params = []
        for a in [x.strip() for x in args.replace("\n", " ").split(",")]:
            if a in ("void", ""):
                continue
            a = re.sub(r"\s+", " ", a)
            if "*" in a:
                params.append("ptr")
            else:
                params.append(a.rsplit(" ", 1)[0].replace("const ", "").strip())     # drop the parameter name
        protos[name] = (re.sub(r"\s+", " ", ret).strip(), params)
    return protos


def test_ctypes_signatures_match_the_header_type_by_type():
    """Every entry of gnan_b200._lib.SIGNATURES against the prototype in the header: same number of parameters, and each scalar type
    of the same width and kind (a 32-bit slot declared for an int64_t argument would pass small values by luck and corrupt large ones)."""
    from gnan_b200 import _lib
    C = ctypes
    scalar = {"int64_t": C.c_int64, "int32_t": C.c_int32, "int": C.c_int, "float": C.c_float, "size_t": C.c_size_t, "uint64_t": C.c_uint64,
              "gnan_stream_t": C.c_void_p}
    protos = _header_prototypes()
    assert sorted(protos) == sorted(_lib.SIGNATURES)
    for name, (res, args) in _lib.SIGNATURES.items():
        ret, params = protos[name]
        assert len(params) == len(args), (name, len(params), len(args))
        for i, (want, got) in enumerate(zip(params, args)):
            if want == "ptr":
                assert got is C.c_void_p or issubclass(got, C._Pointer), (name, i, got)
            else:
                assert got is scalar[want], (name, i, want, got)
        if "*" in ret:
            assert res in (C.c_char_p, C.c_void_p), (name, ret, res)
        else:
            assert res is scalar[ret], (name, ret, res)
