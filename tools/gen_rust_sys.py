#!/usr/bin/env python3
"""Regenerates rust/pcdgpu-sys/src/lib.rs's `extern "C"` block from include/pcdgpu.h (one declaration per exported
function, same order and names).  tests/test_abi_cpu.py checks that the crate declares every function of the header.
  python tools/gen_rust_sys.py            # rewrite
  python tools/gen_rust_sys.py --check    # exit 1 if stale"""
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "rust", "pcdgpu-sys", "src", "lib.rs")
TMAP = {"int": "c_int", "size_t": "usize", "uint32_t": "u32", "uint64_t": "u64", "uint8_t": "u8", "double": "f64",
        "void": "c_void", "char": "c_char"}
HANDLES = {"pcdgpu_ctx", "pcdgpu_bases", "pcdgpu_r1cs", "pcdgpu_pk", "pcdgpu_gm17_pk", "pcdgpu_csr", "pcdgpu_groth16_pvk",
           "pcdgpu_gm17_pvk"}
HEAD = '''// UNCOMPILED SOURCE (see ../../README.md).  The `extern "C"` block is GENERATED from include/pcdgpu.h by
// tools/gen_rust_sys.py: one declaration per exported function, same order, same names.
// Encodings (include/pcdgpu.h): field element = 5 x u64 little-endian Montgomery limbs (ark-ff Fp320 / BigInteger320);
// MSM scalar = 5 x u64 plain (`into_repr()`); affine point = x || y, infinity = all zero; every function returns 0 or
// a negative PCDGPU_E_* code and never unwinds.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] pub struct pcdgpu_ctx { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_bases { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_r1cs { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_pk { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_gm17_pk { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_csr { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_groth16_pvk { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_gm17_pvk { _p: [u8; 0] }

pub const PCDGPU_OK: c_int = 0;
pub const PCDGPU_E_ARG: c_int = -1;
pub const PCDGPU_E_NODEVICE: c_int = -2;
pub const PCDGPU_E_CUDA: c_int = -3;
pub const PCDGPU_E_DOMAIN: c_int = -4;
pub const PCDGPU_E_NOMEM: c_int = -5;
pub const PCDGPU_FIELD_R4: c_int = 0;
pub const PCDGPU_FIELD_Q4: c_int = 1;
pub const PCDGPU_MNT4_298: c_int = 0;
pub const PCDGPU_MNT6_298: c_int = 1;
pub const PCDGPU_MNT4_G1: c_int = 0;
pub const PCDGPU_MNT4_G2: c_int = 1;
pub const PCDGPU_MNT6_G1: c_int = 2;
pub const PCDGPU_MNT6_G2: c_int = 3;
pub const PCDGPU_COMM_ID_BYTES: usize = 128;
pub const PCDGPU_PROF_CLASSES: usize = 11;

#[link(name = "pcdgpu")]
extern "C" {
'''


def conv_type(t):
    t = t.strip()
    const = t.startswith("const ")
    if const:
        t = t[6:].strip()
    stars = t.count("*")
    base = t.replace("*", "").strip()
    out = base if base in HANDLES else TMAP[base]
    for i in range(stars):
        out = ("*const " if (const and i == 0) else "*mut ") + out
    return out


def generate():
    body = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "pcdgpu.h")).read(), flags=re.S)
    decls = re.findall(r"\n((?:const char\*|size_t|int|void)\s+pcdgpu_[a-z0-9_]+\s*\([^;]*\));", body)
    lines = []
    for d in decls:
        d = " ".join(d.split())
        ret, name, args = re.match(r"(const char\*|size_t|int|void)\s+(pcdgpu_[a-z0-9_]+)\s*\((.*)\)$", d).groups()
        params = []
        if args.strip() and args.strip() != "void":
            for a in args.split(","):
                ty, nm = re.match(r"(.*?)([A-Za-z_][A-Za-z0-9_]*)$", a.strip()).groups()
                if nm in ("type", "in", "ref", "fn", "mod", "box"):
                    nm += "_"
                params.append("%s: %s" % (nm, conv_type(ty)))
        r = "" if ret == "void" else (" -> *const c_char" if ret == "const char*" else " -> " + TMAP[ret])
        lines.append("    pub fn %s(%s)%s;" % (name, ", ".join(params), r))
    return HEAD + "\n".join(lines) + "\n}\n"


if __name__ == "__main__":
    text = generate()
    if "--check" in sys.argv:
        sys.exit(0 if open(OUT).read() == text else 1)
    open(OUT, "w").write(text)
