"""dkb_stats has three mirrors besides include/dkb.h: the ctypes Stats of denovo_kmer_b200/_lib.py,
the Rust -sys crate and the dict KmerCounter.stats() returns.  Each must have the C struct's fields
in its order, and the ctypes one its byte layout, or a field read through it comes from another
field's bytes.  CPU only: the offsets come from a C compiler, no library call is made."""
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _c_fields():
    hdr = open(os.path.join(ROOT, "include", "dkb.h")).read()
    body = re.search(r"typedef struct dkb_stats \{(.*?)\} dkb_stats;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = [f.strip() for decl in body.split(";") for f in decl.split(",")]
    return [re.sub(r"^(uint64_t|uint32_t|double|float)\s+", "", f) for f in names if f.strip()]


def test_stats_mirrors_match_the_header(tmp_path):
    from denovo_kmer_b200 import _lib
    c_fields = _c_fields()
    assert c_fields[-2:] == ["occupied_halves", "direct_halves"]
    assert [f for f, _ in _lib.Stats._fields_] == c_fields
    rs = open(os.path.join(ROOT, "bindings", "rust", "denovo-kmer-gpu-sys", "src", "lib.rs")).read()
    rs_body = re.search(r"pub struct DkbStats \{(.*?)\n\}", rs, re.S).group(1)
    assert re.findall(r"pub (\w+):", rs_body) == c_fields
    # byte layout: offsetof / sizeof from gcc against the ctypes structure
    src = tmp_path / "layout.c"
    src.write_text("#include <stddef.h>\n#include <stdio.h>\n#include \"dkb.h\"\nint main(void) {\n" +
                   "".join(f'  printf("{f} %zu\\n", offsetof(dkb_stats, {f}));\n' for f in c_fields) +
                   '  printf("sizeof %zu\\n", sizeof(dkb_stats));\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    want = {f: str(getattr(_lib.Stats, f).offset) for f in c_fields}
    want["sizeof"] = str(__import__("ctypes").sizeof(_lib.Stats))
    assert got == want
