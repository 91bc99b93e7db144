"""Print one kernel's SASS from an object or library, without addresses and symbol names, so
that two builds of a kernel can be diffed instruction for instruction:

    nvcc <flags of denovo_kmer_b200/build.py> -c -o api.o denovo_kmer_b200/csrc/dkb_api.cu
    python scripts/kernel_sass.py old_api.o '_ZN3dkb7k_callsE.*' > old.sass
    python scripts/kernel_sass.py api.o '_ZN3dkb7k_callsILi3EE.*' > new.sass
    diff old.sass new.sass

The second argument is a regular expression for the mangled function name (full match)."""
import re
import subprocess
import sys


def kernel_sass(obj, pattern):
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    for block in re.split(r"\n\s*Function : ", out)[1:]:
        name, body = block.split("\n", 1)
        if re.fullmatch(pattern, name.strip()):
            lines = []
            for line in body.splitlines():
                line = re.sub(r"/\*[0-9a-f]{4}\*/", "", line)  # instruction addresses
                line = re.sub(r"_Z\w+", "<sym>", line)          # symbol names
                if line.strip() and not line.strip().startswith("."):
                    lines.append(line.rstrip())
            return lines
    raise SystemExit(f"no function matching {pattern} in {obj}")


if __name__ == "__main__":
    print("\n".join(kernel_sass(sys.argv[1], sys.argv[2])))
