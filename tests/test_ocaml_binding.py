"""Mechanical consistency checks of the OCaml binding (ocaml/): this image has no OCaml toolchain, so the binding cannot
be compiled for real.  What can be checked without one:
  1. zipc_cuda_stubs.c type-checks with gcc against a minimal mock of the caml/ headers (tests/caml_mock) and the real
     include/zipc_b200.h -- every zipc_b200_* call has the right arity and argument types;
  2. every `external` in zipc_cuda.ml names a CAMLprim stub defined in zipc_cuda_stubs.c with the same number of
     arguments (OCaml externals with more than 5 arguments would need a bytecode twin: there are none);
  3. every `val` declared in zipc_cuda.mli is defined in zipc_cuda.ml, and everything Zipc_deflate's own signature
     (reference src/zipc_deflate.mli) exports has a counterpart;
  4. every function INTEGRATION.md attributes to the OCaml side exists in the .mli."""
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OC = os.path.join(ROOT, "ocaml")


def _read(*p):
    with open(os.path.join(*p)) as f:
        return f.read()


def _strip_ocaml_comments(s):
    out, depth, i = [], 0, 0
    while i < len(s):
        if s.startswith("(*", i):
            depth += 1; i += 2
        elif s.startswith("*)", i) and depth:
            depth -= 1; i += 2
        else:
            if not depth:
                out.append(s[i])
            i += 1
    return "".join(out)


def test_stubs_compile_against_mock_runtime_and_real_header():
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I" + os.path.join(ROOT, "tests", "caml_mock"),
                        "-I" + os.path.join(ROOT, "include"), os.path.join(OC, "zipc_cuda_stubs.c")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def _externals():
    ml = _strip_ocaml_comments(_read(OC, "zipc_cuda.ml"))
    ext = {}
    for m in re.finditer(r"external\s+(\w+)\s*:\s*(.*?)=\s*\"(\w+)\"", ml, re.S):
        name, typ, cname = m.group(1), m.group(2), m.group(3)
        # arity = top-level arrows of the type (tuples/parentheses do not nest arrows here)
        depth, arrows = 0, 0
        for i, ch in enumerate(typ):
            if ch == "(":
                depth += 1
            elif ch == ")":
                depth -= 1
            elif ch == "-" and typ[i:i + 2] == "->" and depth == 0:
                arrows += 1
        ext[name] = (cname, arrows)
    return ext


def test_every_external_has_a_stub_of_the_same_arity():
    stubs = {}
    for m in re.finditer(r"CAMLprim\s+value\s+(\w+)\s*\(([^)]*)\)", _read(OC, "zipc_cuda_stubs.c")):
        stubs[m.group(1)] = len([a for a in m.group(2).split(",") if a.strip()])
    ext = _externals()
    assert len(ext) >= 10
    for name, (cname, arity) in ext.items():
        assert cname in stubs, f"external {name} -> {cname}: no such stub"
        assert stubs[cname] == arity, f"{cname}: OCaml arity {arity}, C arity {stubs[cname]}"
        assert arity <= 5, f"{cname}: more than 5 arguments needs a bytecode stub"
    assert set(stubs) == {c for c, _ in ext.values()}, "stub without an external (or the reverse)"


def test_stub_calls_are_declared_in_the_header():
    hdr = _read(ROOT, "include", "zipc_b200.h")
    declared = set(re.findall(r"\b(zipc_b200_\w+)\s*\(", hdr))
    used = set(re.findall(r"\b(zipc_b200_\w+)\s*\(", _read(OC, "zipc_cuda_stubs.c")))
    assert used and used <= declared, used - declared


def _mli_vals(text):
    return set(re.findall(r"^\s*val\s+(\w+)\s*:", _strip_ocaml_comments(text), re.M))


def test_mli_values_are_defined_and_cover_the_reference_signature():
    mli = _read(OC, "zipc_cuda.mli")
    ml = _strip_ocaml_comments(_read(OC, "zipc_cuda.ml"))
    defined = set(re.findall(r"^\s*(?:let|external|and)\s+(?:rec\s+)?(\w+)", ml, re.M))
    vals = _mli_vals(mli)
    assert vals <= defined, vals - defined
    # the hot-path part of the reference's own signature (src/zipc_deflate.mli of zipc): value names copied here so the
    # test needs nothing outside this repository
    reference = {"equal", "check", "pp", "string", "inflate", "inflate_and_crc_32", "inflate_and_adler_32", "zlib_decompress",
                 "deflate", "crc_32_and_deflate", "adler_32_and_deflate", "zlib_compress"}
    assert reference <= vals
    for batch in ("inflate_batch", "deflate_batch", "strings", "deflate_segmented", "inflate_segmented",
                  "deflate_of_binary_strings", "to_binary_strings", "archive_to_binary_string", "set_device", "set_devices"):
        assert batch in vals, batch


def test_integration_md_names_only_existing_ocaml_functions():
    doc = _read(ROOT, "INTEGRATION.md")
    vals = _mli_vals(_read(OC, "zipc_cuda.mli"))
    named = set(re.findall(r"`(?:Zipc_cuda\.)?(?:File\.)?([a-z_0-9]+)`", doc))
    ocaml_like = {n for n in named if n in {"deflate_segmented", "inflate_segmented", "deflate_of_binary_strings", "to_binary_strings",
                                             "archive_to_binary_string", "inflate_batch", "deflate_batch", "set_device", "set_devices"}}
    assert ocaml_like <= vals, ocaml_like - vals
