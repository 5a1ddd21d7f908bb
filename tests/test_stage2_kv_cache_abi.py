"""CPU checks of the stage-II K/V cache C-ABI: the ctypes mirror of ``cir_stage2_kv_cache`` has the size and field offsets of the C
struct, the ctypes signatures in native.py match the prototypes in include/cir_b200.h, and a C program using them compiles."""
import ctypes as C
import os
import re
import subprocess

import cir_b200 as cir

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ["cir_stage2_kv_cache_bytes", "cir_stage2_kv_cache_init", "cir_stage2_kv_cache_fill",
       "cir_stage2_score_cached_workspace_bytes", "cir_stage2_score_cached"]
STRUCTS = (cir.native.Stage2KVCache, cir.native.Stage2Weights)


def _prototype(name):
    with open(os.path.join(ROOT, "include", "cir_b200.h")) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    m = re.search(r"(\w+)\s+" + name + r"\s*\(([^)]*)\)\s*;", text)
    assert m, name
    return m.group(1), [a.strip() for a in m.group(2).split(",")]


def test_ctypes_signatures_match_the_header():
    sigs = cir.native._SIGS
    for name in NEW:
        ret, args = _prototype(name)
        res, argtypes = sigs[name]
        assert len(args) == len(argtypes), name
        assert res is (C.c_size_t if ret == "size_t" else C.c_int), name
        for decl, t in zip(args, argtypes):
            if "*" in decl:
                assert t is C.c_void_p or (hasattr(t, "_type_") and t._type_ in STRUCTS), (name, decl)
            elif decl.startswith("int64_t"):
                assert t is C.c_int64, (name, decl)
            elif decl.startswith("size_t"):
                assert t is C.c_size_t, (name, decl)
            else:
                raise AssertionError((name, decl))
    assert set(NEW) <= set(cir.native.exported_symbols())


def test_kv_cache_struct_matches_the_c_header(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cir_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(cir_stage2_kv_cache),\n'
                   '  offsetof(cir_stage2_kv_cache, row0), offsetof(cir_stage2_kv_cache, rows), offsetof(cir_stage2_kv_cache, num_tokens),\n'
                   '  offsetof(cir_stage2_kv_cache, dtype), offsetof(cir_stage2_kv_cache, kv)); return 0; }\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    S = cir.native.Stage2KVCache
    assert got == [C.sizeof(S)] + [getattr(S, f).offset for f in ("row0", "rows", "num_tokens", "dtype", "kv")]


def test_new_entry_points_compile_against_the_header(tmp_path):
    src = tmp_path / "use.c"
    src.write_text('#include "cir_b200.h"\n'
                   "int use(cir_ctx* c, const cir_stage2_weights* w, void* blob, const void* tok, const int32_t* i, const void* z,\n"
                   "        float* s, void* ws) {\n"
                   "  cir_stage2_kv_cache kc;\n"
                   "  size_t b = cir_stage2_kv_cache_bytes(c, 10, 577);\n"
                   "  int r = cir_stage2_kv_cache_init(c, blob, b, 0, 10, 577, &kc);\n"
                   "  r += cir_stage2_kv_cache_fill(c, w, &kc, tok, 0, 10);\n"
                   "  size_t n = cir_stage2_score_cached_workspace_bytes(c, 8, 2, 32, kc.num_tokens);\n"
                   "  return r + cir_stage2_score_cached(c, w, &kc, i, 4, z, i, 0, 0, i, 2, 32, i, i, 8, 0, 0, 0, 0, 0, 0, s, 0, ws, n);\n"
                   "}\n")
    subprocess.run(["gcc", "-Wall", "-Werror", "-c", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(tmp_path / "use.o")],
                   check=True)
