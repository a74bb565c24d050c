"""Compare the machine code of two builds of libtvf.so (or of two object files) function by function.

    python tools/compare_sass.py OLD.so NEW.so

Splits `cuobjdump -sass` of each file per kernel and reports the kernels whose instructions (encodings included) differ,
and the kernels only one build has.  Lines that name the file, and the hash in the names of anonymous namespaces, are
ignored.  Exit status 1 if a kernel present in both builds differs.  Builds with the product flags
(tft_vs_fund_b200/build.py) are comparable."""
import re
import subprocess
import sys


def kernels(path):
    """{function name: its SASS lines} of one library or object file."""
    text = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    out, name = {}, None
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", m.group(1))     # the hash follows the source text
            out[name] = []
        elif name is not None and line.strip() and not line.lstrip().startswith(("code for", "Fatbin", "arch =", "host =",
                                                                                  "compile_size", "identifier")):
            out[name].append(line.strip())
    return out


def main(old, new):
    a, b = kernels(old), kernels(new)
    same = [k for k in a if k in b and a[k] == b[k]]
    differ = [k for k in a if k in b and a[k] != b[k]]
    for k in sorted(differ):
        print("DIFFERS   %s" % k)
    for k in sorted(set(a) - set(b)):
        print("REMOVED   %s" % k)
    for k in sorted(set(b) - set(a)):
        print("ADDED     %s" % k)
    print("%d kernels identical, %d differ, %d removed, %d added" % (len(same), len(differ), len(set(a) - set(b)),
                                                                     len(set(b) - set(a))))
    return 1 if differ else 0


if __name__ == "__main__":
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2]))
