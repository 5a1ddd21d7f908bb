"""CPU checks of the C-ABI for re-ranking a device-resident top-K list: the ctypes signatures in native.py match the prototypes in
include/cir_b200.h, the built library exports the symbols, and a C program using the new entry points compiles with -Wall -Werror."""
import ctypes as C
import os
import re
import subprocess

import cir_b200 as cir

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ["cir_stage2_plan_topk", "cir_stage2_rerank_cached_workspace_bytes", "cir_stage2_rerank_cached"]
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


def test_the_library_exports_the_new_symbols():
    out = subprocess.run(["nm", "-D", "--defined-only", cir.native.LIB_PATH], check=True, capture_output=True, text=True).stdout
    exported = {line.split()[-1] for line in out.splitlines() if line.strip()}
    assert set(NEW) <= exported, set(NEW) - exported


def test_new_entry_points_compile_against_the_header(tmp_path):
    src = tmp_path / "use.c"
    src.write_text('#include "cir_b200.h"\n'
                   "int use(cir_ctx* c, const cir_stage2_weights* w, const cir_stage2_kv_cache* kc, const int32_t* cand, const void* z,\n"
                   "        const int32_t* ids, const int32_t* mask, float* s, int32_t* o, int32_t* p, void* ws) {\n"
                   "  int32_t* cnt = p + 4096;\n"
                   "  int r = cir_stage2_plan_topk(c, cand, 4, 50, 32, kc->row0, kc->rows, p, p + 200, p + 400, p + 600, p + 1400, cnt);\n"
                   "  size_t n = cir_stage2_rerank_cached_workspace_bytes(c, 4, 50, 32, kc->num_tokens);\n"
                   "  r += cir_stage2_rerank_cached(c, w, kc, cand, 4, 50, z, ids, mask, 32, s, o, 0, cnt, ws, n);\n"
                   "  return r + cir_stage2_rerank_cached(c, w, kc, cand, 4, 50, z, ids, mask, 32, s, o, p, 0, ws, n);\n"
                   "}\n")
    subprocess.run(["gcc", "-Wall", "-Werror", "-c", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(tmp_path / "use.o")],
                   check=True)
