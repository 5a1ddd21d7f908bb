"""CPU checks of the MXFP8 K/V gallery (CIR_KV_MXFP8): the ctypes signatures in native.py match the prototypes in include/cir_b200.h,
the library exports them, the cache struct keeps its layout, a C program using the new entry points compiles with -Wall -Werror, and
the torch restatement of the quantiser / dequantiser below (which the GPU tests compare the kernels against, bit for bit) follows
the format: power-of-two scale per 32 channels, e4m3 elements rounded to nearest even, exact dequantisation to bf16."""
import ctypes as C
import os
import re
import subprocess

import torch

import cir_b200 as cir

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ["cir_stage2_kv_cache_bytes_mxfp8", "cir_stage2_kv_cache_init_mxfp8", "cir_stage2_kv_cache_fill_mxfp8_workspace_bytes",
       "cir_stage2_kv_cache_fill_mxfp8", "cir_stage2_kv_score_workspace_bytes", "cir_stage2_kv_rerank_workspace_bytes"]
STRUCTS = (cir.native.Stage2KVCache, cir.native.Stage2Weights)
BLOCK, COLS = 32, 3072


# ---------------------------------------------------------------------------------------------------------------- restatement
def mxfp8_scale_exponent(amax: torch.Tensor) -> torch.Tensor:
    """k = max(-127, smallest integer with amax <= 448 * 2^k) per block (amax = 0: -127), int64.  amax = m 2^e, m in [0.5, 1):
    448 2^k = 0.875 2^(k+9), so k = e - 9 when m <= 0.875, else e - 8."""
    m, e = torch.frexp(amax.double())
    k = torch.where(m <= 0.875, e - 9, e - 8).long()
    return torch.where(amax == 0, torch.full_like(k, -127), k.clamp(min=-127))


def mxfp8_quantize(x: torch.Tensor):
    """bf16 K/V rows [R, 3072] -> (e4m3 elements uint8 [R, 3072], E8M0 scales uint8 [R, 96])."""
    assert x.dtype == torch.bfloat16 and x.shape[-1] == COLS
    xb = x.reshape(-1, COLS // BLOCK, BLOCK).double()
    k = mxfp8_scale_exponent(xb.abs().amax(-1))
    y = xb * torch.pow(2.0, (-k).double()).unsqueeze(-1)          # exact: a bf16 value times a power of two, at most 448
    e = y.to(torch.float8_e4m3fn).view(torch.uint8)
    return e.reshape(x.shape), (k + 127).to(torch.uint8).reshape(*x.shape[:-1], COLS // BLOCK)


def mxfp8_dequantize_exact(e: torch.Tensor, s: torch.Tensor) -> torch.Tensor:
    """(elements, scales) -> the float64 values e * 2^k (before any rounding)."""
    v = e.view(torch.float8_e4m3fn).double().reshape(*s.shape, BLOCK)
    return (v * torch.pow(2.0, s.double() - 127).unsqueeze(-1)).reshape(e.shape)


def mxfp8_dequantize(e: torch.Tensor, s: torch.Tensor) -> torch.Tensor:
    """(elements, scales) -> bf16 [R, 3072] = bf16(float(e) * 2^k), what the dequant kernel writes."""
    return mxfp8_dequantize_exact(e, s).to(torch.bfloat16)


def _bits(b: torch.Tensor) -> torch.Tensor:
    return b.view(torch.int16).to(torch.int32) & 0xFFFF


# ---------------------------------------------------------------------------------------------------------------- format
def test_e4m3_cast_rounds_to_nearest_even():
    """The restatement's rounding: every e4m3 value (normal and subnormal) is kept, and a midpoint between two neighbours goes to
    the one with an even code; nothing above the largest midpoint below 448 is fed to the cast."""
    codes = torch.arange(0, 0x7F, dtype=torch.uint8)                          # 0 .. 448 (0x7E); 0x7F is NaN
    vals = codes.view(torch.float8_e4m3fn).double()
    assert vals[0x7E] == 448 and vals[1] == 2.0 ** -9 and vals[8] == 2.0 ** -6      # smallest subnormal, smallest normal
    assert torch.equal(vals.to(torch.float8_e4m3fn).view(torch.uint8), codes)
    mid = (vals[:-1] + vals[1:]) / 2
    got = mid.to(torch.float8_e4m3fn).view(torch.uint8).long()
    lo = codes[:-1].long()
    assert torch.equal(got, torch.where(lo % 2 == 0, lo, lo + 1))
    assert torch.equal((-vals).to(torch.float8_e4m3fn).view(torch.uint8), codes | 0x80)


def test_scale_exponent_matches_the_kernels_bit_formula():
    """The kernel derives the scale byte from the bf16 bits of amax: max(0, E - 8) for mantissa <= 96, else max(0, E - 7)."""
    b = torch.arange(0, 0x7F80, dtype=torch.int32)                             # every finite non-negative bf16
    amax = b.to(torch.int16).view(torch.bfloat16).double()
    E, M = b >> 7, b & 0x7F
    want = torch.where(M <= 96, E - 8, E - 7).clamp(min=0)
    assert torch.equal(mxfp8_scale_exponent(amax) + 127, want.long())
    k = mxfp8_scale_exponent(amax)
    assert bool((amax <= 448 * torch.pow(2.0, k.double())).all())
    smaller = k > -127                                                         # k is the smallest such integer
    assert bool((amax[smaller] > 448 * torch.pow(2.0, k[smaller].double() - 1)).all())


def _block(vals):
    x = torch.zeros(1, COLS, dtype=torch.float64)
    x[0, :len(vals)] = torch.tensor(vals, dtype=torch.float64)
    return x.to(torch.bfloat16)


def test_dequantisation_is_exact_in_bf16():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(64, COLS, generator=g)
    x *= torch.pow(2.0, torch.randint(-140, 120, (64, COLS // BLOCK), generator=g).float()).repeat_interleave(BLOCK, 1)
    x = x.to(torch.bfloat16)
    x[3, 100:140] = 0
    x[5, :64] = -0.0
    e, s = mxfp8_quantize(x)
    exact = mxfp8_dequantize_exact(e, s)
    d = mxfp8_dequantize(e, s)
    assert torch.equal(d.double(), exact)                                     # every e * 2^k is a bf16 value
    assert torch.isfinite(exact).all()
    rel = ((d.double() - x.double()).abs() / x.double().abs().reshape(64, -1, BLOCK).amax(-1).repeat_interleave(BLOCK, 1).clamp(min=1e-300))
    assert float(rel.max()) <= 2.0 ** -4 + 1e-12                             # half an e4m3 ulp of the block maximum at most


def test_block_edge_cases():
    # amax exactly 448 * 2^k: k itself, the element 448 (0x7E), no rounding up to the next scale
    for k in (-20, 0, 3, 100):
        e, s = mxfp8_quantize(_block([448 * 2.0 ** k, -(2.0 ** k)]))
        assert s[0, 0] == k + 127 and e[0, 0] == 0x7E and e[0, 1] == 0xB8, (k, s[0, 0], e[0, :2])
        assert torch.equal(mxfp8_dequantize(e, s)[0, :2], _block([448 * 2.0 ** k, -(2.0 ** k)])[0, :2])
    # just above 448 * 2^k (450, the next bf16 value): the next exponent
    e, s = mxfp8_quantize(_block([450.0]))
    assert s[0, 0] == 128 and e[0, 0] == 0x76                                 # 225 -> 224 = 1.75 * 2^7
    # an all-zero block: k = -127, zero elements; -0.0 keeps its sign through both directions
    e, s = mxfp8_quantize(_block([0.0, -0.0]))
    assert (s == 0).all() and e[0, 0] == 0x00 and e[0, 1] == 0x80 and (e[0, 2:] == 0).all()
    d = mxfp8_dequantize(e, s)
    assert _bits(d[0, :2]).tolist() == [0x0000, 0x8000]
    # e4m3 subnormals: elements below 2^-6 of the scaled block, rounded to multiples of 2^-9
    e, s = mxfp8_quantize(_block([448.0, 2.0 ** -9, 3 * 2.0 ** -9, 2.0 ** -10, 3 * 2.0 ** -11, 2.0 ** -7 + 2.0 ** -9]))
    assert s[0, 0] == 127
    assert e[0, :6].tolist() == [0x7E, 0x01, 0x03, 0x00, 0x01, 0x05]        # 2^-10 ties to 0 (even), 1.5 * 2^-10 rounds to 2^-9
    # tiny amax: k clamps at -127 and the block keeps its bf16 values exactly (they are multiples of 2^-133)
    tiny = [2.0 ** -130, -3 * 2.0 ** -133, 2.0 ** -126, 5 * 2.0 ** -128]
    x = _block(tiny)
    e, s = mxfp8_quantize(x)
    assert s[0, 0] == 0
    assert torch.equal(mxfp8_dequantize(e, s), x)


# ---------------------------------------------------------------------------------------------------------------- ABI
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


def test_format_constant_and_unchanged_struct(tmp_path):
    with open(os.path.join(ROOT, "include", "cir_b200.h")) as f:
        text = f.read()
    assert re.search(r"#define CIR_KV_MXFP8 2\b", text) and cir.native.KV_MXFP8 == 2
    assert {cir.native.DTYPE_F32, cir.native.DTYPE_BF16}.isdisjoint({cir.native.KV_MXFP8})
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cir_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(cir_stage2_kv_cache),\n'
                   '  offsetof(cir_stage2_kv_cache, row0), offsetof(cir_stage2_kv_cache, rows), offsetof(cir_stage2_kv_cache, num_tokens),\n'
                   '  offsetof(cir_stage2_kv_cache, dtype), offsetof(cir_stage2_kv_cache, kv)); return 0; }\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [40, 0, 8, 16, 24, 32]                                      # the layout of the bf16 cache's release
    S = cir.native.Stage2KVCache
    assert got == [C.sizeof(S)] + [getattr(S, f).offset for f in ("row0", "rows", "num_tokens", "dtype", "kv")]


def test_cache_bytes():
    """12 layers x rows x N x (3072 element bytes + 96 scale bytes), 256-byte aligned: 21.93 MB per image at N = 577."""
    lib = cir.native.lib()
    assert lib.cir_stage2_kv_cache_bytes_mxfp8(None, 1, 577) == -(-12 * 577 * 3168 // 256) * 256
    assert abs(lib.cir_stage2_kv_cache_bytes_mxfp8(None, 1000, 577) / 1000 / 1e6 - 21.93) < 0.01
    assert lib.cir_stage2_kv_cache_bytes_mxfp8(None, -1, 577) == 0


def test_new_entry_points_compile_against_the_header(tmp_path):
    src = tmp_path / "use.c"
    src.write_text('#include "cir_b200.h"\n'
                   "int use(cir_ctx* c, const cir_stage2_weights* w, void* blob, const void* tok, const int32_t* i, const void* z,\n"
                   "        float* s, int32_t* o, void* ws) {\n"
                   "  cir_stage2_kv_cache kc;\n"
                   "  size_t b = cir_stage2_kv_cache_bytes_mxfp8(c, 10, 577);\n"
                   "  int r = cir_stage2_kv_cache_init_mxfp8(c, blob, b, 0, 10, 577, &kc);\n"
                   "  size_t f = cir_stage2_kv_cache_fill_mxfp8_workspace_bytes(c, &kc, 4);\n"
                   "  r += cir_stage2_kv_cache_fill_mxfp8(c, w, &kc, tok, 0, 10, ws, f);\n"
                   "  r += kc.dtype == CIR_KV_MXFP8 ? 0 : 1;\n"
                   "  size_t n = cir_stage2_kv_score_workspace_bytes(c, &kc, 8, 4, 2, 32);\n"
                   "  r += cir_stage2_score_cached(c, w, &kc, i, 4, z, i, 0, 0, i, 2, 32, i, i, 8, 0, 0, 0, 0, 0, 0, s, 0, ws, n);\n"
                   "  n = cir_stage2_kv_rerank_workspace_bytes(c, &kc, 4, 50, 32);\n"
                   "  return r + cir_stage2_rerank_cached(c, w, &kc, i, 4, 50, z, i, i, 32, s, o, 0, 0, ws, n);\n"
                   "}\n")
    subprocess.run(["gcc", "-Wall", "-Werror", "-c", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(tmp_path / "use.o")],
                   check=True)
