"""CPU checks of the compaction / id-search C-ABI: the ctypes signatures in native.py match the prototypes in include/cir_b200.h, and
a C program that calls the new entry points with the header's types compiles."""
import ctypes as C
import os
import re
import subprocess

import cir_b200 as cir

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ["cir_stage1_index_compact_workspace_bytes", "cir_stage1_index_compact",
       "cir_stage1_index_topk_ids_workspace_bytes", "cir_stage1_index_topk_ids"]


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
                assert t is C.c_void_p or (hasattr(t, "_type_") and t._type_ is cir.native.Stage1Index), (name, decl)
            elif decl.startswith("int64_t"):
                assert t is C.c_int64, (name, decl)
            elif decl.startswith("uint32_t"):
                assert t is C.c_uint32, (name, decl)
            elif decl.startswith("size_t"):
                assert t is C.c_size_t, (name, decl)
            else:
                raise AssertionError((name, decl))
    assert set(NEW) <= set(cir.native.exported_symbols())


def test_new_entry_points_compile_against_the_header(tmp_path):
    src = tmp_path / "use.c"
    src.write_text('#include "cir_b200.h"\n'
                   "int use(cir_ctx* c, cir_stage1_index* s, cir_stage1_index* d, const float* q, const int32_t* ids, uint32_t* t,\n"
                   "        int32_t* di, float* td, int32_t* ti, void* ws) {\n"
                   "  size_t a = cir_stage1_index_compact_workspace_bytes(c, s);\n"
                   "  size_t b = cir_stage1_index_topk_ids_workspace_bytes(c, s, 4, 10);\n"
                   "  int r = cir_stage1_index_compact(c, s, t, ids, 0xFFFFFFFFu, d, t, di, ws, a);\n"
                   "  return r + cir_stage1_index_topk_ids(c, d, q, 4, di, 100, 0, 0, 0, 0, 10, td, ti, 0, ws, b);\n"
                   "}\n")
    subprocess.run(["gcc", "-Wall", "-Werror", "-c", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(tmp_path / "use.o")],
                   check=True)
