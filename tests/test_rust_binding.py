"""rust/ (the UNCOMPILED Rust side of the boundary) against include/gaast_b200.h, without a Rust
toolchain: the sys crate's extern block symbol by symbol, its #[repr(C)] structs and constants, and
that the patches apply to the reference (`git apply --check` on a scratch copy)."""
import ctypes as C
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "gaast_b200.h")
LIB_RS = os.path.join(ROOT, "rust", "gaast-b200-sys", "src", "lib.rs")
PATCHES = os.path.join(ROOT, "rust", "patches")

SCALARS = {"int": "c_int", "int32_t": "i32", "uint32_t": "u32", "uint64_t": "u64", "uint16_t": "u16", "size_t": "usize", "double": "f64",
           "float": "f32", "void": "c_void", "char": "c_char", "unsigned char": "u8", "gaast_status": "c_int"}


def _c_type_to_rust(t: str) -> str:
    """'const gaast_batch* const*' -> '*const *const gaast_batch' (pointer levels right to left)."""
    t = " ".join(t.replace("*", " * ").split())
    toks = t.split(" ")
    base, i = [], 0
    while i < len(toks) and toks[i] != "*":
        base.append(toks[i])
        i += 1
    const_base = "const" in base
    name = " ".join(x for x in base if x != "const")
    rust = SCALARS.get(name, name)
    levels = []  # per '*': whether what it points to is const
    pointee_const = const_base
    while i < len(toks):
        assert toks[i] == "*", t
        i += 1
        ptr_const = False
        if i < len(toks) and toks[i] == "const":
            ptr_const = True
            i += 1
        levels.append(pointee_const)
        pointee_const = ptr_const
    for c in levels:
        rust = ("*const " if c else "*mut ") + rust
    return rust


def _header_prototypes():
    h = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    out = {}
    for ret, name, args in re.findall(r"^([A-Za-z_][\w\s\*]*?[\s\*])(gaast_\w+)\s*\(([^;{]*?)\)\s*;", h, flags=re.M):
        params = []
        args = " ".join(args.split())
        if args != "void":
            for a in args.split(","):
                m = re.match(r"^(.*?)(\w+)$", a.strip())  # strip the parameter name
                params.append(_c_type_to_rust(m.group(1).strip()))
        ret = ret.strip()
        out[name] = (None if ret == "void" else _c_type_to_rust(ret), params)
    return out


def _rust_prototypes():
    src = open(LIB_RS).read()
    block = src[src.index('extern "C" {'):]
    out = {}
    for name, args, ret in re.findall(r"pub fn (gaast_\w+)\(([^)]*)\)\s*(?:->\s*([^;]+))?;", block):
        params = [a.split(":", 1)[1].strip() for a in (x.strip() for x in args.split(",")) if a]
        out[name] = (ret.strip() if ret else None, params)
    return out


def test_c_type_translation():
    assert _c_type_to_rust("gaast_batch* const*") == "*const *mut gaast_batch"
    assert _c_type_to_rust("const double* const*") == "*const *const f64"
    assert _c_type_to_rust("void* const*") == "*const *mut c_void"
    assert _c_type_to_rust("gaast_ctx**") == "*mut *mut gaast_ctx"
    assert _c_type_to_rust("const char*") == "*const c_char"
    assert _c_type_to_rust("uint64_t") == "u64"


def test_extern_block_matches_the_header_symbol_by_symbol():
    want, got = _header_prototypes(), _rust_prototypes()
    assert len(want) >= 46
    assert sorted(want) == sorted(got), (sorted(set(want) - set(got)), sorted(set(got) - set(want)))
    for name in want:
        assert got[name] == want[name], f"{name}: rust {got[name]} vs header {want[name]}"


def test_every_bound_symbol_is_exported_by_the_library():
    from gaast_b200 import _lib as L
    for name in _rust_prototypes():
        assert hasattr(L.lib, name), name


def _rust_structs():
    src = open(LIB_RS).read()
    out = {}
    for name, body in re.findall(r"#\[repr\(C\)\][^{]*?pub struct (\w+)\s*\{(.*?)\n\}", src, flags=re.S):
        out[name] = [(f, t.strip()) for f, t in re.findall(r"pub (\w+):\s*([^,\n]+),", body)]
    return out


def _header_structs():
    h = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    out = {}
    for body, name in re.findall(r"typedef struct \w+\s*\{(.*?)\}\s*(\w+);", h, flags=re.S):
        fields = []
        for decl in [d.strip() for d in body.split(";") if d.strip()]:
            m = re.match(r"^(.*?)(\w+)$", decl)
            fields.append((m.group(2), _c_type_to_rust(m.group(1).strip())))
        out[name] = fields
    return out


RUST_SIZES = {"u16": 2, "u32": 4, "u64": 8, "f64": 8, "f32": 4, "usize": 8}


def _size(fields):
    off, align = 0, 1
    for _, t in fields:
        s = 8 if t.startswith("*") else RUST_SIZES[t]
        off = (off + s - 1) // s * s + s
        align = max(align, s)
    return (off + align - 1) // align * align


def test_repr_c_structs_match_the_header():
    from gaast_b200 import _lib as L
    want, got = _header_structs(), _rust_structs()
    assert sorted(want) == sorted(got) == ["gaast_input_desc", "gaast_op", "gaast_plan_desc", "gaast_term"]
    for name in want:
        assert got[name] == want[name], f"{name}: rust {got[name]} vs header {want[name]}"
    for name, ct in (("gaast_term", L.Term), ("gaast_op", L.Op), ("gaast_input_desc", L.InputDesc), ("gaast_plan_desc", L.PlanDesc)):
        assert _size(got[name]) == C.sizeof(ct), name
    assert [_size(got[n]) for n in ("gaast_term", "gaast_op", "gaast_input_desc", "gaast_plan_desc")] == [16, 32, 16, 88]


def test_constants_match_the_header():
    h = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    src = open(LIB_RS).read()
    rust = {k: int(v) for k, v in re.findall(r"pub const (GAAST_\w+):\s*\w+\s*=\s*(\d+);", src)}
    enums = {k: int(v) for k, v in re.findall(r"\b(GAAST_\w+)\s*=\s*(\d+)", h)}
    defines = {k: int(v) for k, v in re.findall(r"#define (GAAST_\w+)\s+(\d+)u", h)}
    assert len(enums) >= 20 and len(defines) == 2
    for name, val in {**enums, **defines}.items():
        assert rust.get(name) == val, f"{name}: rust {rust.get(name)} vs header {val}"


def test_patches_apply_to_the_reference(tmp_path):
    """Needs a checkout of the reference (github.com/YPares/gaast), named by GAAST_REFERENCE_DIR.

    The repository does not ship the reference.  To make this test self-contained, store the six files the patches
    touch (Cargo.toml, src/ast/mod.rs, src/ast/specialize.rs, src/graded.rs, src/eval.rs, src/lib.rs) under
    tests/golden/, use them when GAAST_REFERENCE_DIR is unset, and check each file's `git hash-object` against the
    abbreviated pre-image blob id on the `index` line of the patch that touches it, so that the stored copies are
    known to be the reference's own."""
    ref = os.environ.get("GAAST_REFERENCE_DIR", "")
    if not os.path.isdir(os.path.join(ref, "src")):
        pytest.skip("GAAST_REFERENCE_DIR does not name a checkout of the reference")
    dst = tmp_path / "gaast"
    shutil.copytree(ref, dst, ignore=shutil.ignore_patterns(".git"))
    patches = sorted(os.path.join(PATCHES, p) for p in os.listdir(PATCHES) if p.endswith(".patch"))
    assert len(patches) == 5
    for p in patches:
        r = subprocess.run(["git", "apply", "--check", p], cwd=dst, capture_output=True, text=True)
        assert r.returncode == 0, f"{os.path.basename(p)}: {r.stderr}"
        subprocess.run(["git", "apply", p], cwd=dst, check=True)
    assert "pub fn lower(&self) -> Result<FlatPlan, LowerError>" in open(dst / "src" / "ast" / "specialize.rs").read()
    assert "pub fn eval_batch" in open(dst / "src" / "eval.rs").read()
    assert "pub struct DeviceBatch" in open(dst / "src" / "graded.rs").read()
    assert 'cuda = ["eval", "dep:gaast-b200-sys"]' in open(dst / "Cargo.toml").read()
