"""Regenerates tests/golden/* from a checkout of the reference (zipc):
    python tests/golden/make_golden.py <zipc checkout>/test/test.ml

zip-docs.zip is the fixture embedded as an OCaml string literal in the reference's
test/test.ml:131-3294 (Info-ZIP made; 1 dir + 2 deflate members).  The literal
consists only of \\xHH escapes and line continuations; it is decoded here and its fingerprint
checked against SURVEY.md section 8c (56,924 bytes, CRC-32 0a88d91b, md5 d2076f2e...).
"""
import hashlib
import os
import re
import sys
import zlib

HERE = os.path.dirname(os.path.abspath(__file__))


def extract_fixture(ref_test: str) -> bytes:
    src = open(ref_test, "rb").read().decode("latin-1")
    start = src.index("zip_docs_zip :=")
    lit_start = src.index('"', start) + 1
    lit_end = src.index('"', lit_start)
    lit = src[lit_start:lit_end]
    lit = re.sub(r"\\\n[ \t]*", "", lit)  # OCaml line continuation: backslash newline blanks
    assert re.fullmatch(r"(\\x[0-9a-fA-F]{2})*", lit), "unexpected escape in fixture literal"
    return bytes(int(h, 16) for h in re.findall(r"\\x([0-9a-fA-F]{2})", lit))


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    data = extract_fixture(sys.argv[1])
    assert len(data) == 56924, len(data)
    assert zlib.crc32(data) == 0x0A88D91B, hex(zlib.crc32(data))
    assert hashlib.md5(data).hexdigest() == "d2076f2e591c1af277938f79485fe0d7"
    with open(os.path.join(HERE, "zip-docs.zip"), "wb") as f:
        f.write(data)
    print("zip-docs.zip", len(data), "bytes ok")


if __name__ == "__main__":
    main()
