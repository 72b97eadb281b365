"""Generates integration/rust/zkb200-sys/src/lib.rs (extern "C" declarations + ffi_wrap) from include/zkb200.h, so the Rust
binding a zktls maintainer would add (INTEGRATION.md) never drifts from the C-ABI.  There is no Rust toolchain in this image:
the output is source only; tests/test_abi_symbols.py checks that it is current and covers every declared symbol."""
import os, re, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TYPES = {"int": "c_int", "size_t": "usize", "uint32_t": "u32", "uint64_t": "u64", "float": "f32", "char": "c_char", "void": "c_void",
         "zkb_ctx": "ZkbCtx", "zkb_prover": "ZkbProver", "zkb_program": "ZkbProgram",
         "zkb_session": "ZkbSession"}


def rust_type(ctype):
    ctype = ctype.strip()
    stars = ctype.count("*")
    const = "const" in ctype.split("*")[0]
    base = ctype.replace("const", "").replace("*", "").strip()
    r = TYPES[base]
    for _ in range(stars):
        r = ("*const " if const else "*mut ") + r
        const = False if stars > 1 else const
    return r


def parse(header):
    text = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    out = []
    for m in re.finditer(r"(zkb_err|const char\*|void)\s+(zkb_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", text):
        ret, name, args = m.group(1), m.group(2), m.group(3).strip()
        params = []
        if args and args != "void":
            for a in args.split(","):
                a = " ".join(a.split())
                mm = re.match(r"(.*?)(\w+)$", a)
                params.append((mm.group(2), rust_type(mm.group(1))))
        out.append((name, ret, params))
    return out


def generate():
    fns = parse(open(os.path.join(ROOT, "include", "zkb200.h")).read())
    lines = ["//! zkb200-sys: raw bindings to libzkb200.so (GENERATED from include/zkb200.h by tools/gen_rust_ffi.py -- do not edit).",
             "//! Conventions are those of risc0-sys: every operator returns NULL or a malloc'd message (`ffi_wrap`).",
             "#![allow(non_camel_case_types)]", "use std::ffi::{c_char, c_int, c_void, CStr};", "",
             "#[repr(C)] pub struct ZkbCtx { _private: [u8; 0] }", "#[repr(C)] pub struct ZkbProver { _private: [u8; 0] }",
             "#[repr(C)] pub struct ZkbProgram { _private: [u8; 0] }", "#[repr(C)] pub struct ZkbSession { _private: [u8; 0] }",
             "pub type ZkbErr = *const c_char;", "", '#[link(name = "zkb200")]', 'extern "C" {']
    for name, ret, params in fns:
        r = {"zkb_err": " -> ZkbErr", "const char*": " -> *const c_char", "void": ""}[ret]
        lines.append(f"    pub fn {name}({', '.join(f'{n}: {t}' for n, t in params)}){r};")
    lines += ["}", "",
              "/// NULL = Ok; otherwise copy the message, free it with zkb_free_error and return it as an error (risc0-sys `ffi_wrap`).",
              "pub fn ffi_wrap<F: FnOnce() -> ZkbErr>(f: F) -> Result<(), String> {",
              "    let e = f();", "    if e.is_null() { return Ok(()); }",
              "    let msg = unsafe { CStr::from_ptr(e) }.to_string_lossy().into_owned();",
              "    unsafe { zkb_free_error(e) };", "    Err(msg)", "}", ""]
    return "\n".join(lines), [f[0] for f in fns]


if __name__ == "__main__":
    src, names = generate()
    path = os.path.join(ROOT, "integration", "rust", "zkb200-sys", "src", "lib.rs")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    open(path, "w").write(src)
    print(path, len(names), "functions")
