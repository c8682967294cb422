"""CPU tests of the drop-in boundary: the shared library loads, exports every symbol that
include/erirt_b200.h declares, and fails loudly (no CPU fallback) when no GPU is present."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "erirt_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(erirt_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from erirt_b200 import _lib
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    from erirt_b200 import _lib
    declared = _declared_symbols()
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/erirt_b200.h but not exported"
    assert sorted(_lib.EXPORTED) == declared
    assert lib.erirt_version() == _lib.ABI_VERSION


def test_config_struct_matches_header(lib):
    from erirt_b200 import _lib
    # field order and sizes of erirt_config as laid out by the C compiler
    assert ctypes.sizeof(_lib.Config) == 144 and ctypes.sizeof(_lib.Stats) == 48
    assert _lib.Config.q_rt.offset == 56 and _lib.Config.seed.offset == 80 and _lib.Config.nu_cell_moments.offset == 112 and _lib.Config.reserved.offset == 116


def test_no_cpu_fallback(lib):
    """Without a CUDA device every compute entry point must fail with ERIRT_E_CUDA, not compute on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import erirt_b200 as E
    with pytest.raises(E.ErirtError) as ei:
        E.Engine("RtIrtNull", 10, 3, 0)
    assert ei.value.code == -2 and "no CPU fallback" in str(ei.value)
    with pytest.raises(E.ErirtError):
        E.k_pg(np.zeros((2, 2)))
    with pytest.raises(E.ErirtError):
        E.k_philox([0] * 4, [0] * 2)


def test_argument_validation_happens_before_cuda(lib):
    import erirt_b200 as E
    with pytest.raises(ValueError, match="item type must be '1pl' or '2pl'"):
        E.Engine("RtIrt", 10, 3, 1, itemtype="3pl")
    with pytest.raises(E.ErirtError) as ei:
        E.Engine("RtIrt", 10, 3, 1, q_rt=1.5)
    assert ei.value.code == -1
    with pytest.raises(E.ErirtError) as ei:
        E.Engine("RtIrt", 0, 3, 1)
    assert ei.value.code == -1


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure: nothing in the package may reference it."""
    pkg = os.path.join(ROOT, "extendedrtirtmodeling.jl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle_py" not in txt and "liberirt_oracle" not in txt and "import oracle" not in txt, f


def test_environment_and_build_switches_are_the_documented_ones():
    """The ERIRT_* environment variables the product reads are exactly those of the table in INTEGRATION.md section 5, and the only
    ERIRT_* macros the kernels test with #if / #ifdef / #ifndef are the three diagnostic builds: no tuning switch selects a path
    that the benchmark does not run."""
    pkg = os.path.join(ROOT, "extendedrtirtmodeling.jl_b200")
    sources = [os.path.join(ROOT, "bench.py")]
    sources += [os.path.join(ROOT, "julia", f) for f in os.listdir(os.path.join(ROOT, "julia")) if f.endswith(".jl")]
    for dirpath, _, files in os.walk(pkg):
        sources += [os.path.join(dirpath, f) for f in files if f.endswith((".py", ".cu", ".cuh", ".h"))]
    read = set()
    for path in sources:
        txt = open(path, encoding="utf-8", errors="ignore").read()
        read |= set(re.findall(r'(?:getenv\(|os\.environ\.get\(|get\(ENV,\s*)"(ERIRT_[A-Z0-9_]+)"', txt))
    doc = open(os.path.join(ROOT, "INTEGRATION.md"), encoding="utf-8").read()
    table = doc[doc.index("## 5. Environment switches"):]
    table = table[:table.index("\n## ")] if "\n## " in table else table
    documented = set(re.findall(r"^\|\s*`(ERIRT_[A-Z0-9_]+)`\s*\|", table, flags=re.M))
    assert read == documented, f"read but not documented: {sorted(read - documented)}; documented but not read: {sorted(documented - read)}"

    tested = set()
    for dirpath, _, files in os.walk(os.path.join(pkg, "csrc")):
        for f in files:
            for line in open(os.path.join(dirpath, f), encoding="utf-8", errors="ignore"):
                if re.match(r"\s*#\s*(?:if|ifdef|ifndef)\b", line):
                    tested |= set(re.findall(r"\b(ERIRT_[A-Z0-9_]+)\b", line))
    assert tested == {"ERIRT_TICKS", "ERIRT_TIMELINE", "ERIRT_CHECKS"}, sorted(tested)


def test_julia_stub_matches_the_header(lib):
    """julia/ErirtB200.jl cannot be executed here (no Julia): check statically that its ErirtConfig mirrors erirt_config field by field
    (names, order, widths) and that every C symbol it ccalls is declared in include/erirt_b200.h."""
    import re
    from erirt_b200 import _lib
    src = open(os.path.join(ROOT, "julia", "ErirtB200.jl"), encoding="utf-8").read()
    body = src[src.index("struct ErirtConfig"):]
    body = body[:body.index("\nend")]
    fields = re.findall(r"^\s+(\w+)::([\w{},]+)\s*$", body, flags=re.M)
    jl_size = {"Int32": 4, "UInt32": 4, "Int64": 8, "UInt64": 8, "Float64": 8}
    assert [f for f, _ in fields] == [f[0] for f in _lib.Config._fields_]
    for (name, jt), cf in zip(fields, _lib.Config._fields_):
        m = re.fullmatch(r"NTuple\{(\d+),(\w+)\}", jt)
        size = int(m.group(1)) * jl_size[m.group(2)] if m else jl_size[jt]
        assert size == ctypes.sizeof(cf[1]), (name, jt)
    called = set(re.findall(r"ccall\(\(:(\w+), LIB\)", src))
    assert called and called <= set(_declared_symbols()), called - set(_declared_symbols())
    assert {"erirt_create", "erirt_set_data", "erirt_set_data_y8", "erirt_set_state", "erirt_sample", "erirt_get_trace", "erirt_get_moments",
            "erirt_destroy", "erirt_generate_data", "erirt_checkpoint_save", "erirt_checkpoint_load", "erirt_comm_init", "erirt_peer_export",
            "erirt_peer_attach", "erirt_peer_detach", "erirt_trace_width"} <= called
    # large-N and sharded entry points exist (VERDICT r1 item 10)
    for needle in ("mutable struct LeanPost", "function lean(", "sample!(MCMC::LeanGibbs", "sample_sharded!", "person_trace_fits"):
        assert needle in src, needle


def _c_prototypes():
    """name -> (return type, [argument types]) of every function declared in include/erirt_b200.h (comments stripped)."""
    src = open(os.path.join(ROOT, "include", "erirt_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    protos = {}
    for m in re.finditer(r"(?:^|\n)\s*((?:const\s+)?[a-z0-9_]+\s*\**)\s*(erirt_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", src):
        ret, name, args = m.group(1), m.group(2), m.group(3)
        types = []
        for a in [x.strip() for x in args.split(",")]:
            if a in ("", "void"):
                continue
            a = re.sub(r"\[\d*\]", "*", a)                  # array parameters decay to pointers
            stars = a.count("*")
            words = [w for w in re.sub(r"\*", " ", a).split() if w != "const"]
            base = words[0] if len(words) == 1 or words[0] not in ("unsigned",) else " ".join(words[:2])
            types.append(base + "*" * stars)
        protos[name] = (re.sub(r"\s+", "", ret.replace("const", "")), types)
    return protos


def test_julia_ccall_signatures_match_the_header(lib):
    """Every ccall of julia/ErirtB200.jl passes the number and the kinds of arguments the C prototype declares, and reads the return
    value with the right width (the stub cannot be executed here, so this is the static check that stands in for running it)."""
    protos = _c_prototypes()
    assert len(protos) >= 25
    ok = {"erirt_handle*": {"Ptr{Cvoid}"}, "erirt_handle**": {"Ref{Ptr{Cvoid}}"}, "erirt_config*": {"Ref{ErirtConfig}"},
          "double*": {"Ptr{Float64}"}, "uint8_t*": {"Ptr{Bool}", "Ptr{UInt8}"}, "void*": {"Ptr{UInt8}", "Ptr{Cvoid}"},
          "int64_t": {"Int64"}, "int32_t": {"Int32", "Cint"}, "uint64_t": {"UInt64"}, "uint32_t": {"UInt32"}, "erirt_stats*": {"Ref{ErirtStats}"}}
    ret_ok = {"int": {"Cint", "Int32"}, "int64_t": {"Int64"}, "char*": {"Cstring"}}
    src = open(os.path.join(ROOT, "julia", "ErirtB200.jl"), encoding="utf-8").read()
    calls = re.findall(r"ccall\(\(:(\w+), LIB\),\s*(\w+),\s*\(([^)]*)\)", src, flags=re.S)
    assert len(calls) >= 15
    for name, ret, args in calls:
        cret, cargs = protos[name]
        jargs = [a.strip() for a in args.split(",") if a.strip()]
        assert ret in ret_ok[cret], (name, "return", ret, cret)
        assert len(jargs) == len(cargs), (name, jargs, cargs)
        for ja, ca in zip(jargs, cargs):
            assert ja in ok[ca], (name, ja, ca)
