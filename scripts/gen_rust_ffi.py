#!/usr/bin/env python
"""Generates rust/src/ffi.rs (the `extern "C"` block and #[repr(C)] structs) from include/fd_b200.h, so the Rust side of
the boundary cannot drift from the header: tests/test_abi.py regenerates it and compares with the committed file.

    python scripts/gen_rust_ffi.py            # rewrite rust/src/ffi.rs
    python scripts/gen_rust_ffi.py --check    # exit 1 if the committed file is stale
"""
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "fd_b200.h")
OUT = os.path.join(ROOT, "rust", "src", "ffi.rs")

PRIM = {"int": "c_int", "int32_t": "i32", "int64_t": "i64", "uint8_t": "u8", "uint32_t": "u32", "float": "f32", "double": "f64",
        "size_t": "usize", "void": "c_void", "char": "c_char", "unsigned": "c_uint"}


def strip_comments(src):
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return re.sub(r"//[^\n]*", "", src)


def rust_type(ctype, consts):
    """'const float *const *' -> '*const *const f32'; plain names map through PRIM or stay (struct names)."""
    toks = re.findall(r"[A-Za-z_][A-Za-z0-9_]*|\*", ctype)
    base, i = None, 0
    quals = []          # const flag pending for the next level
    const_base = False
    while i < len(toks) and toks[i] != "*":
        if toks[i] == "const":
            const_base = True
        elif toks[i] not in ("struct", "enum"):
            base = toks[i]
        i += 1
    t = PRIM.get(base, base)
    const_next = const_base
    while i < len(toks):
        if toks[i] == "*":
            t = ("*const " if const_next else "*mut ") + t
            const_next = False
        elif toks[i] == "const":
            # `T *const` qualifies the pointer just emitted: affects the NEXT level's pointee constness
            const_next = True
        i += 1
    return t


def split_params(s):
    out, depth, cur = [], 0, ""
    for ch in s:
        if ch in "([":
            depth += 1
        elif ch in ")]":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur.strip())
            cur = ""
        else:
            cur += ch
    if cur.strip():
        out.append(cur.strip())
    return out


RESERVED = {"box", "in", "type", "ref", "fn", "mod", "use", "loop", "match", "move", "self", "super", "where", "as"}


def parse_param(p, consts):
    m = re.match(r"^(.*)\(\s*\*\s*([A-Za-z_][A-Za-z0-9_]*)\s*\)\s*\[\s*(\w+)\s*\]$", p)   # const int64_t (*shape)[4]
    if m:
        inner = rust_type(m.group(1).replace("const", "").strip(), consts)
        n = consts.get(m.group(3), m.group(3))
        const = "const" in m.group(1)
        return m.group(2), "%s [%s; %s]" % ("*const" if const else "*mut", inner, n)
    m = re.match(r"^(.*?)([A-Za-z_][A-Za-z0-9_]*)$", p)
    ctype, name = m.group(1).strip(), m.group(2)
    if not ctype:                       # unnamed parameter (e.g. `void`)
        return None, rust_type(name, consts)
    if name in RESERVED:
        name += "_"
    return name, rust_type(ctype, consts)


def parse_header(src):
    src = strip_comments(src)
    consts = dict(re.findall(r"#define\s+(FD_[A-Z_]+)\s+(\d+)", src))
    enums = []
    for m in re.finditer(r"typedef\s+enum\s+\w+\s*\{(.*?)\}\s*(\w+)\s*;", src, flags=re.S):
        enums.append((m.group(2), [(k, int(v)) for k, v in re.findall(r"(\w+)\s*=\s*(\d+)", m.group(1))]))
    for m in re.finditer(r"(?<!typedef\s)enum\s*\{(.*?)\}\s*;", src, flags=re.S):
        enums.append((None, [(k, int(v)) for k, v in re.findall(r"(\w+)\s*=\s*(\d+)", m.group(1))]))
    structs = [(m.group(3), parse_fields(m.group(2), consts))
               for m in re.finditer(r"typedef\s+struct\s+(\w+)\s*\{(.*?)\}\s*(\w+)\s*;", src, flags=re.S)]
    # `typedef struct X X;` names an opaque type unless `struct X {...};` defines it (parse_plain_structs)
    defined = {name for name, _ in parse_plain_structs(src)}
    opaque = [o for o in re.findall(r"typedef\s+struct\s+(\w+)\s+(\w+)\s*;", src) if o[0] not in defined]
    body = re.sub(r"typedef\s+(struct|enum)\s+\w+\s*\{.*?\}\s*\w+\s*;", "", src, flags=re.S)
    body = re.sub(r"(?<!typedef\s)struct\s+\w+\s*\{.*?\}\s*;", "", body, flags=re.S)
    body = re.sub(r"enum\s*\{.*?\}\s*;", "", body, flags=re.S)
    body = re.sub(r"typedef[^;]*;", "", body)
    body = re.sub(r"#[^\n]*", "", body)
    body = body.replace('extern "C" {', "").replace("}", "")
    funcs = []
    for stmt in body.split(";"):
        stmt = " ".join(stmt.split())
        m = re.match(r"^(.*?)([A-Za-z_][A-Za-z0-9_]*)\s*\((.*)\)$", stmt)
        if not m:
            continue
        ret, name, params = m.group(1).strip(), m.group(2), m.group(3).strip()
        plist = [] if params in ("", "void") else [parse_param(p, consts) for p in split_params(params)]
        funcs.append((name, ret, plist))
    return consts, enums, structs, [o[1] for o in opaque], funcs


def parse_plain_structs(src):
    """structs defined as `struct X {...};` and named by a separate `typedef struct X X;` -> [(name, fields)]"""
    src = strip_comments(src)
    consts = dict(re.findall(r"#define\s+(FD_[A-Z_]+)\s+(\d+)", src))
    return [(m.group(1), parse_fields(m.group(2), consts))
            for m in re.finditer(r"(?<!typedef\s)struct\s+(\w+)\s*\{(.*?)\}\s*;", src, flags=re.S)]


def parse_fields(body, consts):
    """the field declarations of one struct body -> [(name, rust type)]"""
    fields = []
    for decl in body.split(";"):
        decl = " ".join(decl.split())
        if not decl:
            continue
        first, *rest = split_params(decl)
        fm = re.match(r"^(.*?)([A-Za-z_][A-Za-z0-9_]*)((?:\s*\[\s*\w+\s*\])*)$", first)
        ctype_full = fm.group(1).strip()
        base = ctype_full.replace("*", "").strip()
        for d in [fm.group(2) + fm.group(3)] + [r.strip() for r in rest]:
            stars = d.count("*") + (ctype_full.count("*") if d == fm.group(2) + fm.group(3) else 0)
            dm = re.match(r"^\**\s*([A-Za-z_][A-Za-z0-9_]*)((?:\s*\[\s*\w+\s*\])*)$", d.replace(" ", ""))
            name, dims = dm.group(1), re.findall(r"\[\s*(\w+)\s*\]", dm.group(2))
            t = rust_type(base + " " + "*" * stars, consts)
            for n in reversed(dims):
                t = "[%s; %s]" % (t, n if not n.isdigit() else n)
            fields.append((name, t))
    return fields


def generate():
    src = open(HEADER).read()
    consts, enums, structs, opaque, funcs = parse_header(src)
    structs = structs + parse_plain_structs(src)
    o = []
    o.append("//! src/ffi.rs — `extern \"C\"` declarations of include/fd_b200.h (the only unsafe surface of the crate).")
    o.append("//! Replaces the commented-out binding in src/rcnn/gpu_nms.rs:9-19.")
    o.append("//! GENERATED by scripts/gen_rust_ffi.py from include/fd_b200.h — do not edit (tests/test_abi.py checks it is current).")
    o.append("#![allow(non_camel_case_types, non_upper_case_globals, non_snake_case, dead_code)]")
    o.append("use std::os::raw::{c_char, c_int, c_void};")
    o.append("")
    for k, v in consts.items():
        o.append("pub const %s: usize = %s;" % (k, v))
    o.append("")
    for name, items in enums:
        if name:
            o.append("pub type %s = c_int;" % name)
        for k, v in items:
            o.append("pub const %s: c_int = %d;" % (k, v))
        o.append("")
    for name in opaque:
        o.append("#[repr(C)]")
        o.append("pub struct %s { _private: [u8; 0] }" % name)
    o.append("")
    for name, fields in structs:
        o.append("#[repr(C)]")
        o.append("#[derive(Clone, Copy)]")
        o.append("pub struct %s {" % name)
        for fname, ftype in fields:
            o.append("    pub %s: %s," % (fname, ftype))
        o.append("}")
    o.append("")
    o.append("extern \"C\" {")
    for name, ret, plist in funcs:
        args = ", ".join("%s: %s" % (n or "_a%d" % i, t) for i, (n, t) in enumerate(plist))
        r = "" if ret == "void" else " -> " + rust_type(ret, consts)
        o.append("    pub fn %s(%s)%s;" % (name, args, r))
    o.append("}")
    o.append("")
    o.append("/// Maps an fd_status to the crate's error type (the reference bubbles `anyhow::Error`, e.g. face_detection.rs:135-138).")
    o.append("pub fn check(rc: c_int) -> anyhow::Result<()> {")
    o.append("    if rc == 0 { return Ok(()); }")
    o.append("    let msg = unsafe { std::ffi::CStr::from_ptr(fd_last_error()) }.to_string_lossy().into_owned();")
    o.append("    Err(anyhow::anyhow!(\"fd_b200 error {}: {}\", rc, msg))")
    o.append("}")
    return "\n".join(o) + "\n"


if __name__ == "__main__":
    text = generate()
    if "--check" in sys.argv:
        sys.exit(0 if os.path.exists(OUT) and open(OUT).read() == text else 1)
    open(OUT, "w").write(text)
    print(OUT)
