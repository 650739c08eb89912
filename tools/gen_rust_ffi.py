#!/usr/bin/env python3
"""Prints the Rust `extern "C"` block for every function include/zkpair.h declares (the `src/ffi.rs` of
INTEGRATION.md section 3 is generated with this; tests/test_host_logic.py checks that it stays complete)."""
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TYPES = [
    (r"^zkp_ctx \*\*$", "*mut *mut ZkpCtx"), (r"^const zkp_ctx \*$", "*const ZkpCtx"), (r"^zkp_ctx \*$", "*mut ZkpCtx"),
    (r"^zkp_groth16_vk \*\*$", "*mut *mut ZkpGroth16Vk"), (r"^const zkp_groth16_vk \*$", "*const ZkpGroth16Vk"),
    (r"^zkp_groth16_vk \*$", "*mut ZkpGroth16Vk"),
    (r"^zkp_kzg_setup \*\*$", "*mut *mut ZkpKzgSetup"), (r"^const zkp_kzg_setup \*$", "*const ZkpKzgSetup"),
    (r"^zkp_kzg_setup \*$", "*mut ZkpKzgSetup"),
    (r"^const uint64_t \*$", "*const u64"), (r"^uint64_t \*$", "*mut u64"), (r"^const uint8_t \*$", "*const u8"),
    (r"^uint8_t \*$", "*mut u8"), (r"^const uint32_t \*$", "*const u32"), (r"^uint32_t \*$", "*mut u32"), (r"^uint32_t$", "u32"), (r"^const void \*$", "*const c_void"),
    (r"^void \*$", "*mut c_void"), (r"^const int \*$", "*const c_int"), (r"^double \*$", "*mut f64"),
    (r"^const char \*$", "*const c_char"), (r"^size_t$", "usize"), (r"^int32_t$", "i32"), (r"^uint64_t$", "u64"),
    (r"^int$", "c_int"), (r"^void$", "()"),
]


def rust_type(c):
    c = re.sub(r"\s+", " ", c.strip())
    for pat, r in TYPES:
        if re.match(pat, c):
            return r
    raise SystemExit("unmapped C type: %r" % c)


def declarations():
    hdr = open(os.path.join(ROOT, "include", "zkpair.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    for m in re.finditer(r"^([\w ]+?\*?)\s*\b(zkp_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", hdr, flags=re.M):
        ret, name, args = m.group(1), m.group(2), m.group(3)
        ret = ret.strip()
        if name + "(" in hdr and ret:
            params = []
            if args.strip() not in ("", "void"):
                for a in args.split(","):
                    a = re.sub(r"\s+", " ", a.strip())
                    mm = re.match(r"^(.*?)(\w+)$", a)
                    params.append((mm.group(2), rust_type(mm.group(1))))
            yield name, params, rust_type(ret)


def main():
    out = ["extern \"C\" {"]
    for name, params, ret in declarations():
        sig = ", ".join("%s: %s" % (("r#%s" % n) if n in ("in", "type") else n, t) for n, t in params)
        line = "    pub fn %s(%s)%s;" % (name, sig, "" if ret == "()" else " -> " + ret)
        out.append(line)
    out.append("}")
    print("\n".join(out))


if __name__ == "__main__":
    main()
