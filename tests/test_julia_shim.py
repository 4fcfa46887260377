"""julia/SDPLRPlusB200.jl cannot be executed here (no Julia toolchain).  What CAN be pinned without one: every `ccall` of the
shim names an entry point that include/sdplrp_b200.h declares, with the same number of arguments and compatible scalar
types, and the shim's mirrors of the native structs match the header field for field."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

C2J = {"int32_t": {"Int32", "Cint"}, "int64_t": {"Int64"}, "uint64_t": {"UInt64"}, "double": {"Float64"}}


def header_prototypes():
    src = open(os.path.join(ROOT, "include", "sdplrp_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
    protos = {}
    for m in re.finditer(r"\b(?:int32_t|const char \*|void \*)\s*(sdplrp_\w+)\s*\(([^;{]*?)\)\s*;", src, flags=re.S):
        args = [a.strip() for a in m.group(2).split(",")] if m.group(2).strip() not in ("", "void") else []
        protos[m.group(1)] = args
    return protos


def split_top(s):
    out, depth, cur = [], 0, ""
    for ch in s:
        if ch in "({[":
            depth += 1
        elif ch in ")}]":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur.strip()); cur = ""
        else:
            cur += ch
    if cur.strip():
        out.append(cur.strip())
    return out


def shim_ccalls():
    src = open(os.path.join(ROOT, "julia", "SDPLRPlusB200.jl")).read()
    calls = []
    for m in re.finditer(r"ccall\(\(:(\w+), LIB\),\s*(\w+),\s*\(", src):
        i, depth = m.end(), 1
        while depth:
            depth += {"(": 1, ")": -1}.get(src[i], 0)
            i += 1
        calls.append((m.group(1), m.group(2), split_top(src[m.end():i - 1])))
    return calls


def test_every_ccall_matches_the_header():
    protos = header_prototypes()
    calls = shim_ccalls()
    assert len(calls) >= 25
    for name, ret, jargs in calls:
        assert name in protos, f"{name} is not declared in include/sdplrp_b200.h"
        cargs = protos[name]
        assert len(jargs) == len(cargs), f"{name}: {len(jargs)} Julia argument types vs {len(cargs)} in the header ({cargs})"
        for j, c in zip(jargs, cargs):
            pointer_c = "*" in c or "[" in c
            pointer_j = j.startswith(("Ptr{", "Ref{")) or j == "Cstring"
            assert pointer_c == pointer_j, f"{name}: {j} vs {c}"
            if not pointer_c:
                ctype = c.replace("const", "").split()[0]
                assert j in C2J[ctype], f"{name}: {j} vs {c}"
            elif "double" in c:
                assert "Float64" in j, f"{name}: {j} vs {c}"
            elif "int64_t" in c:
                assert "Int64" in j, f"{name}: {j} vs {c}"


def test_native_structs_mirror_the_header_field_for_field():
    hdr = open(os.path.join(ROOT, "include", "sdplrp_b200.h")).read()
    jl = open(os.path.join(ROOT, "julia", "SDPLRPlusB200.jl")).read()

    def c_fields(struct_name):
        body = re.search(r"typedef struct \{([^}]*)\} " + struct_name + ";", hdr).group(1)
        body = re.sub(r"/\*.*?\*/", " ", body, flags=re.S)
        names = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            names += [re.sub(r"\[.*\]", "", x).strip() for x in decl.split(None, 1)[1].split(",")]
        return names

    def j_fields(struct_name):
        body = re.search(r"struct " + struct_name + r"\n(.*?)\nend", jl, flags=re.S).group(1)
        return [f.split("::")[0].strip() for part in body.split("\n") for f in part.split(";") if "::" in f]

    assert j_fields("NativeConfig") == c_fields("sdplrp_config")
    assert j_fields("NativeResult") == c_fields("sdplrp_result")


def test_mode_fields_are_compared_as_symbols():
    """BurerMonteiroConfig stores gtol_mode / ptol_mode / objtol_mode as Symbols (src/options.jl:21-23)."""
    jl = open(os.path.join(ROOT, "julia", "SDPLRPlusB200.jl")).read()
    assert '== "relative"' not in jl
    assert jl.count("== :relative") >= 5
