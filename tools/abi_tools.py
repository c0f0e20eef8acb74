"""Parses the C ABI (include/multilinear_b200.h) and the Rust extern block (rust/cuda.rs) into comparable signatures, and
generates the extern block from the header so the two cannot drift (tests/test_abi.py compares them).

    python tools/abi_tools.py --write     # regenerate the block between the GENERATED markers of rust/cuda.rs
"""
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HANDLES = {"ml_transcript": "MlTranscript", "ml_merkle": "MlMerkle", "ml_fri": "MlFri", "ml_fri_proof": "MlFriProof", "ml_sumcheck": "MlSumcheck",
           "ml_wsumcheck": "MlWSumcheck", "ml_pcs_proof": "MlPcsProof", "ml_bfri_proof": "MlBfriProof", "ml_bpcs_proof": "MlBpcsProof",
           "ml_shard": "MlShard", "ml_bfri": "MlBfri", "ml_pcs_shard": "MlPcsShard", "ml_bpcs_shard": "MlBpcsShard",
           "ml_wsumcheck_shard": "MlWSumcheckShard", "ml_fri_shard": "MlFriShard", "ml_bfri_shard": "MlBfriShard"}
SCALARS = {"int": "c_int", "unsigned": "c_uint", "size_t": "usize", "uint64_t": "u64", "int64_t": "i64", "uint32_t": "u32", "uint8_t": "u8",
           "double": "f64", "char": "c_char", "void": "c_void"}
BEGIN, END = "    // ---- GENERATED from include/multilinear_b200.h by tools/abi_tools.py (do not edit by hand)\n", "    // ---- END GENERATED\n"


def c_type_to_rust(ctype):
    """'const uint8_t *const *' -> '*const *const u8'; arrays were rewritten to pointers by the caller"""
    t = ctype.strip()
    # split into base (with its const) and pointer levels (each possibly const)
    m = re.match(r"^(const\s+)?(\w+)\s*(.*)$", t)
    if not m:
        raise ValueError(ctype)
    base_const, base, rest = bool(m.group(1)), m.group(2), m.group(3).replace(" ", "")
    if base in HANDLES:
        rust = HANDLES[base]
    elif base in SCALARS:
        rust = SCALARS[base]
    else:
        raise ValueError("unknown C type %r" % ctype)
    levels = re.findall(r"\*(const)?", rest)
    if not levels:
        assert not base_const, ctype
        return rust
    # innermost pointer's constness is the base's const; outer levels: the const written AFTER the inner '*' qualifies that pointer
    # C: T *const *p  ->  p: pointer to (const pointer to T)  ->  Rust *const *mut T
    quals = [base_const] + [lv == "const" for lv in levels[:-1]]
    out = rust
    for q in quals:
        out = ("*const " if q else "*mut ") + out
    return out


def parse_header(path=None):
    text = open(path or os.path.join(ROOT, "include", "multilinear_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"^\s*#.*$", "", text, flags=re.M)
    sigs = {}
    for m in re.finditer(r"([\w\s\*]+?)\b(ml_[a-z0-9_]+)\s*\(([^;{}]*?)\)\s*;", text):
        ret, name, args = m.group(1).strip(), m.group(2), m.group(3).strip()
        if ret.startswith("typedef") or "extern" in ret:
            continue
        rargs = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                arr = re.match(r"^(.*?)(\w+)\s*\[\s*\d*\s*\]$", a)  # `const uint8_t gen[16]` decays to a pointer
                if arr:
                    ty, nm = arr.group(1).strip() + " *", arr.group(2)
                else:
                    mm = re.match(r"^(.*?)(\w+)$", a)
                    ty, nm = mm.group(1).strip(), mm.group(2)
                rargs.append((nm, c_type_to_rust(ty)))
        rret = None if ret == "void" else c_type_to_rust(ret)
        sigs[name] = (rargs, rret)
    return sigs


RUST_KEYWORDS = {"gen": "gen_", "in": "in_", "type": "type_", "ref": "ref_", "fn": "fn_", "box": "box_"}


def rust_extern_block(sigs):
    lines = [BEGIN]
    for name in sorted(sigs):
        args, ret = sigs[name]
        a = ", ".join("%s: %s" % (RUST_KEYWORDS.get(n, n), t) for n, t in args)
        lines.append("    pub fn %s(%s)%s;\n" % (name, a, "" if ret is None else " -> " + ret))
    lines.append(END)
    return "".join(lines)


def parse_rust(path=None):
    text = open(path or os.path.join(ROOT, "rust", "cuda.rs")).read()
    text = re.sub(r"//.*$", "", text, flags=re.M)
    sigs = {}
    for blk in re.finditer(r'extern\s+"C"\s*\{(.*?)\n\}', text, flags=re.S):
        for m in re.finditer(r"pub\s+fn\s+(ml_[a-z0-9_]+)\s*\((.*?)\)\s*(?:->\s*([^;]+?))?\s*;", blk.group(1), flags=re.S):
            name, args, ret = m.group(1), m.group(2).strip(), (m.group(3) or "").strip() or None
            rargs = []
            if args:
                for a in args.split(","):
                    n, t = a.split(":", 1)
                    rargs.append((n.strip(), " ".join(t.split())))
            sigs[name] = (rargs, ret)
    return sigs


def main(argv):
    sigs = parse_header()
    block = rust_extern_block(sigs)
    if "--write" in argv:
        p = os.path.join(ROOT, "rust", "cuda.rs")
        s = open(p).read()
        i, j = s.index(BEGIN), s.index(END) + len(END)
        open(p, "w").write(s[:i] + block + s[j:])
        print("rust/cuda.rs: %d declarations regenerated" % len(sigs))
    else:
        sys.stdout.write(block)
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
