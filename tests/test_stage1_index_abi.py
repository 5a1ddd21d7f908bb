"""CPU checks of the resident stage-I index binding: the ctypes mirror of ``cir_stage1_index`` has the size of the C struct."""
import ctypes as C
import os
import subprocess

import cir_b200 as cir

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_stage1_index_struct_matches_the_c_header(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "cir_b200.h"\n'
                   'int main(void) { printf("%zu\\n", sizeof(cir_stage1_index)); return 0; }\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    size = int(subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout)
    assert size == C.sizeof(cir.native.Stage1Index)
