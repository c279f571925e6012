"""Compare the SASS of two builds of the library, kernel by kernel (no GPU needed).

    python tools/sass_compare.py OLD.so NEW.so [-v NAME_SUBSTRING]

Prints how many kernels of OLD compile to identical instructions in NEW, and names the differing, missing and new ones.
Addresses and the per-file header lines (source path, architecture) are left out of the comparison.  -v prints the
first lines of the diff of the first differing kernel whose name contains NAME_SUBSTRING.  Exit code 1 if a kernel of
OLD differs or is missing.
"""
import difflib
import re
import subprocess
import sys

_HEADER = re.compile(r"(Fatbin|code for|\.target|identifier|arch =|code version|host =|compile_size|\.section|=+$)")


def kernels(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    d, name, buf = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                d[name] = buf
            name, buf = m.group(1), []
            continue
        if name is not None:
            t = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).strip()
            if t and not _HEADER.match(t):
                buf.append(t)
    if name:
        d[name] = buf
    return d


def main():
    a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
    same = [k for k in a if k in b and a[k] == b[k]]
    diff = [k for k in a if k in b and a[k] != b[k]]
    gone = [k for k in a if k not in b]
    new = [k for k in b if k not in a]
    print("old kernels %d: identical %d, differing %d, missing %d; new kernels %d" % (len(a), len(same), len(diff), len(gone),
                                                                                     len(new)))
    for tag, names in (("DIFF", diff), ("GONE", gone), ("NEW ", new)):
        for k in names:
            print(tag, k)
    if "-v" in sys.argv:
        pick = [k for k in diff if sys.argv[sys.argv.index("-v") + 1] in k]
        if pick:
            for line in list(difflib.unified_diff(a[pick[0]], b[pick[0]], lineterm=""))[:40]:
                print(line)
    return 1 if diff or gone else 0


if __name__ == "__main__":
    sys.exit(main())
