"""CPU: the C-ABI library loads and exports every symbol include/*.h declares; without a GPU it fails loudly (no CPU fallback)."""
import ctypes as C
import os
import re

import pytest

from kolibrie_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    names = set()
    for hdr in ("kolibrie_b200.h", "cudajoin.h"):
        text = open(os.path.join(ROOT, "include", hdr)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        names |= set(re.findall(r"\b(kb_[a-z0-9_]+|perform_hash_join_cuda)\s*\(", text))
    names -= {"kb_filter_opcode"}
    return names


def test_library_exports_every_declared_symbol():
    L = C.CDLL(capi.LIB_PATH)
    decl = declared_symbols()
    assert len(decl) >= 39
    for name in sorted(decl):
        assert hasattr(L, name), f"{name} declared in include/ but not exported"
    assert set(capi.EXPORTED_SYMBOLS) == decl


def test_legacy_alias_library_exports_the_reference_symbol():
    """Kolibrie links `cudajoin` (kolibrie/build.rs:75-79) and binds perform_hash_join_cuda (cuda_join.rs:14-26)."""
    L = C.CDLL(capi.LEGACY_LIB_PATH)
    assert hasattr(L, "perform_hash_join_cuda")


def test_version_and_loud_failure_without_gpu():
    L = capi.lib()
    assert b"sm_100a" in L.kb_version()
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(capi.KolibrieError) as e:
        capi.Context(0)
    assert "no CPU fallback" in str(e.value)


def test_struct_layouts_match_header():
    assert C.sizeof(capi.KbTerm) == 8 and C.sizeof(capi.KbPattern) == 24 and C.sizeof(capi.KbFilterOp) == 24
    assert C.sizeof(capi.KbAgg) == 8 and C.sizeof(capi.KbRuleFilter) == 24 and C.sizeof(capi.KbRule) == 48
    assert C.sizeof(capi.KbFixpointStats) == 8 + 8 + 8 + 64 * 8 + 8
    assert capi.lib().kb_shard_of(12345, 8) < 8


def test_every_entry_point_is_documented_for_the_integrator():
    """INTEGRATION.md is the binding guide: every function the header declares must at least be named there"""
    import re

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "kolibrie_b200.h")).read()
    doc = open(os.path.join(root, "INTEGRATION.md")).read()
    fns = re.findall(r"KB_API\s+[\w\s\*]+?\b(kb_\w+)\s*\(", header)
    assert len(fns) >= 45
    names = set(re.findall(r"kb_\w+", doc))
    # `kb_groups_info/keys/values/counts/free` style lists name a family by its prefix
    for fam in re.findall(r"(kb_\w+?_)(\w+(?:/\w+)+)", doc):
        for tail in fam[1].split("/"):
            names.add(fam[0] + tail)
    missing = [f for f in fns if f not in names]
    assert not missing, missing


def test_ctypes_signatures_match_the_header():
    """every kb_* function the Python binding declares (capi.lib(): argtypes / restype) against the header: same number of parameters,
    the same scalar width where the header passes a scalar, a pointer where it passes a pointer — a 32-bit argument where the callee
    reads 64 bits (or the reverse) is the ABI bug this guards against"""
    from tests.test_rust_shim_ffi import header_functions

    L = capi.lib()
    hdr = header_functions()
    scalars = {"u32": (C.c_uint32,), "u64": (C.c_uint64,), "i32": (C.c_int32, C.c_int), "f64": (C.c_double,), "u8": (C.c_uint8,)}
    checked = 0
    for name, (ret, args) in sorted(hdr.items()):
        fn = getattr(L, name)
        if fn.argtypes is None:
            continue  # not declared by the binding (it declares what it calls)
        assert len(fn.argtypes) == len(args), f"{name}: {len(fn.argtypes)} argtypes, {len(args)} parameters in the header"
        for i, (at, (base, levels)) in enumerate(zip(fn.argtypes, args)):
            if levels:
                assert at is C.c_void_p or at is C.c_char_p or hasattr(at, "contents") or issubclass(at, C._Pointer), f"{name} parameter {i}: {at} for a pointer"
            else:
                assert at in scalars[base], f"{name} parameter {i}: {at} for a {base}"
        rbase, rlevels = ret
        if rlevels:
            assert fn.restype in (C.c_void_p, C.c_char_p) or issubclass(fn.restype, C._Pointer), f"{name}: result {fn.restype}"
        elif rbase == "void":
            assert fn.restype is None, f"{name}: result {fn.restype} for void"
        else:
            assert fn.restype in scalars[rbase], f"{name}: result {fn.restype} for {rbase}"
        checked += 1
    assert checked >= 60, checked


def test_legacy_header_is_the_signature_kolibrie_binds():
    """include/cudajoin.h against the definition it replaces (kolibrie/src/cuda/cuda_join.cu:48-56) and the Rust declaration that calls it
    (cuda_join.rs:14-26): parameter for parameter. Both parameter lists are stored in tests/golden/reference/cuda_join_signature.json."""
    import json

    from tests.golden.reference.make_reference_golden import c_params

    with open(os.path.join(ROOT, "tests", "golden", "reference", "cuda_join_signature.json")) as f:
        ref = json.load(f)
    ours = c_params(open(os.path.join(ROOT, "include", "cudajoin.h")).read(), "void perform_hash_join_cuda(")
    theirs = ref["cuda_join.cu"]
    assert ours == theirs, (ours, theirs)
    rust = ref["cuda_join.rs"]
    assert [x.split(":")[0].strip() for x in rust] == [re.findall(r"\w+", x)[-1] for x in ours]
    depth = lambda t: t.count("*")
    assert [depth(x.split(":")[1]) for x in rust] == [depth(x) for x in ours], "pointer depth per parameter as Rust passes it"


def test_the_product_never_touches_the_oracle():
    """the oracle is test infrastructure: nothing under kolibrie_b200/ imports it or the tests package, the shared library neither links
    it nor carries its symbols nor any math / BLAS / thrust dependency beyond the C++ runtime, and bench.py reaches it only from inside the
    functions of its CPU legs (cpu baseline, reference arm, the other configs' CPU samples) — never at module level"""
    import ast
    import subprocess

    pkg = os.path.join(ROOT, "kolibrie_b200")
    for d, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith(".py"):
                tree = ast.parse(open(os.path.join(d, f)).read())
                for node in ast.walk(tree):
                    names = [a.name for a in node.names] if isinstance(node, ast.Import) else [node.module or ""] if isinstance(node, ast.ImportFrom) else []
                    for n in names:
                        assert not re.match(r"^(tests|oracle)(\.|$)", n), f"{f} imports {n}"
            if f.endswith((".cu", ".cuh", ".hpp", ".h")):
                text = open(os.path.join(d, f), errors="replace").read()
                assert not re.search(r'#include\s+[<"][^>"]*oracle', text), f
    needed = subprocess.run(["readelf", "-d", capi.LIB_PATH], stdout=subprocess.PIPE, text=True).stdout
    libs = set(re.findall(r"NEEDED\)\s+Shared library: \[([^\]]+)\]", needed))
    assert libs <= {"libstdc++.so.6", "libm.so.6", "libgcc_s.so.1", "libc.so.6", "ld-linux-x86-64.so.2", "libdl.so.2", "libpthread.so.0", "librt.so.1"}, libs
    syms = subprocess.run(["nm", "-D", "--defined-only", capi.LIB_PATH], stdout=subprocess.PIPE, text=True).stdout
    assert not re.search(r"\bko_\w+", syms), "oracle symbols inside the product library"
    bench = ast.parse(open(os.path.join(ROOT, "bench.py")).read())
    for node in bench.body:  # module level only
        if isinstance(node, (ast.Import, ast.ImportFrom)):
            mod = node.module if isinstance(node, ast.ImportFrom) else ",".join(a.name for a in node.names)
            assert "oracle" not in (mod or "") and not (mod or "").startswith("tests"), mod
