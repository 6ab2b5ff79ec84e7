"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol include/porrt_b200.h
declares (no compute calls -- there is no GPU here), and the product fails loudly without a device."""
import glob
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "porrt_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(porrt_[a-z0-9_]+)\s*\(", src)))


def _ensure_built():
    so = os.path.join(ROOT, "po_rrt_b200", "libporrt_b200.so")
    if not os.path.exists(so):
        subprocess.run(["make", "-C", os.path.join(ROOT, "po_rrt_b200", "csrc"), "-j4"], check=True, capture_output=True)
    return so


def test_header_is_plain_c():
    subprocess.run(["gcc", "-std=c99", "-fsyntax-only", "-x", "c", os.path.join(ROOT, "include", "porrt_b200.h")], check=True)


def test_library_exports_every_declared_symbol():
    so = _ensure_built()
    out = subprocess.run(["nm", "-D", "--defined-only", so], check=True, capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (porrt_[a-z0-9_]+)", out))
    declared = _declared_symbols()
    assert len(declared) >= 25
    missing = [s for s in declared if s not in exported]
    assert not missing, "declared in include/porrt_b200.h but not exported: %s" % missing


def test_ctypes_signatures_cover_header():
    from po_rrt_b200 import _lib
    _ensure_built()
    _lib.load()  # AttributeError if a typed symbol is missing from the .so
    assert sorted(_lib.SIGNATURES) == _declared_symbols()


def test_sm100a_code_present():
    so = _ensure_built()
    out = subprocess.run(["cuobjdump", "--list-elf", so], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_no_cpu_fallback():
    import torch
    import po_rrt_b200 as P
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    _ensure_built()
    with pytest.raises(P.PorrtError):
        P.Context()


def test_product_does_not_touch_oracle():
    pkg = os.path.join(ROOT, "po_rrt_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", "Makefile")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "pyoracle" not in text and "liboracle" not in text and "porrt_oracle" not in text, f


def test_rust_ffi_is_generated_from_header():
    """integration/rust/src/b200_ffi.rs (the crate-side `extern "C"` block, INTEGRATION.md) binds exactly what
    include/porrt_b200.h declares and is what scripts/gen_rust_ffi.py produces from the header today"""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import gen_rust_ffi
    text = open(gen_rust_ffi.OUT).read()
    assert text == gen_rust_ffi.render(), "stale: run python scripts/gen_rust_ffi.py"
    missing = [s for s in _declared_symbols() if ("pub fn %s(" % s) not in text]
    assert not missing, missing


def test_rust_integration_files_use_only_declared_symbols():
    """the hand-written Rust half (feature-gated impls, planner-level swaps) calls nothing the header does not declare"""
    rust_dir = os.path.join(ROOT, "integration", "rust")
    declared = set(_declared_symbols())
    used = set()
    for dirpath, _, files in os.walk(rust_dir):
        for f in files:
            if f.endswith(".rs") and f != "b200_ffi.rs":
                used |= set(re.findall(r"\b(porrt_[a-z0-9_]+)\s*\(", open(os.path.join(dirpath, f)).read()))
    assert used <= declared, sorted(used - declared)


def test_rust_build_script_lists_the_makefile_sources():
    """integration/rust/build.rs compiles exactly the translation units of po_rrt_b200/csrc/Makefile (and watches its headers)"""
    mk = open(os.path.join(ROOT, "po_rrt_b200", "csrc", "Makefile")).read()
    srcs = re.search(r"^SRCS := (.*)$", mk, flags=re.M).group(1).split()
    hdrs = re.search(r"^%\.o: %\.cu (.*)$", mk, flags=re.M).group(1).split()
    rs = open(os.path.join(ROOT, "integration", "rust", "build.rs")).read()
    listed = re.findall(r'"([a-z0-9_]+\.cu)"', rs)
    assert sorted(listed) == sorted(srcs)
    for h in hdrs:
        if h.startswith(".."):
            continue
        assert '"%s"' % h in rs, h
    for f in ("b200_ffi.rs", "b200.rs", "prm_b200.rs", "qmdp_b200.rs", "pto_b200.rs", "refiner_b200.rs"):
        assert os.path.exists(os.path.join(ROOT, "integration", "rust", "src", f))
    # every library function the hand-written Rust files call is declared in the generated FFI block
    ffi = open(os.path.join(ROOT, "integration", "rust", "src", "b200_ffi.rs")).read()
    for f in ("b200.rs", "prm_b200.rs", "qmdp_b200.rs", "pto_b200.rs", "refiner_b200.rs"):
        src = open(os.path.join(ROOT, "integration", "rust", "src", f)).read()
        for name in sorted(set(re.findall(r"\b(porrt_[a-z0-9_]+)\s*\(", src))):
            assert ("pub fn %s(" % name) in ffi, (f, name)


# DESIGN.md 0: no run-time backend switch and no environment variable that selects an implementation.  The CUDA sources read
# PORRT_DEBUG (diagnostic prints) and PORRT_NCCL_LIB (where NCCL is loaded from, include/porrt_b200.h) and nothing else, and no
# `#ifndef` leaves a constant open to a -D override; paths that tests must reach on inputs where the library would not choose them
# are context options (PORRT_OPT_FORCE_*).
def _csrc_without_comments():
    paths = sorted(glob.glob(os.path.join(ROOT, "po_rrt_b200", "csrc", "*.cu*")))
    assert paths
    for p in paths:
        src = re.sub(r"/\*.*?\*/", "", open(p).read(), flags=re.S)
        yield os.path.basename(p), re.sub(r"//[^\n]*", "", src)


def test_library_reads_only_documented_environment_variables():
    allowed = {"PORRT_DEBUG", "PORRT_NCCL_LIB"}
    found = [(name, m.group(1).strip()) for name, src in _csrc_without_comments() for m in re.finditer(r"\bgetenv\s*\(([^)]*)\)", src)]
    assert found
    bad = [(name, arg) for name, arg in found if not arg.startswith('"') or arg.strip('"') not in allowed]
    assert not bad, "environment variables read by the library beyond %s: %s" % (sorted(allowed), bad)


def test_work_space_is_carved_from_named_buffers():
    # every block of work space is laid out once (Carve, common.cuh) in a buffer with a name and listed users, not by a bump lambda
    # of its own or in a numbered slot whose owner nothing records
    bad = []
    for name, src in _csrc_without_comments():
        bad += [(name, m.group(0)) for m in re.finditer(r"\b(?:scratch|pin)\s*\[\s*\d+\s*\]|\bauto\s+take\w*\s*=\s*\[", src)]
    assert not bad, "numbered work-space slots or hand-written take lambdas: %s" % bad


def test_library_has_no_ifndef_knobs():
    # an include guard is `#ifndef X` directly followed by a bare `#define X`; anything else is a compile-time knob
    bad = []
    for name, src in _csrc_without_comments():
        lines = [l.strip() for l in src.splitlines() if l.strip()]
        for i, l in enumerate(lines):
            m = re.match(r"#\s*ifndef\s+(\w+)$", l)
            if m and not (i + 1 < len(lines) and re.fullmatch(r"#\s*define\s+%s" % m.group(1), lines[i + 1])):
                bad.append((name, m.group(1)))
    assert not bad, "#ifndef knobs in the library sources: %s" % bad
