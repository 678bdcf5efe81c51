"""Per-kernel SASS of two builds of libnig_b200.so: every kernel of the first must have the identical instruction stream in
the second (cuobjdump -sass; addresses, encodings and line info stripped). Exit status 1 if one differs or is missing.

    python tools/sass_compare.py <parent libnig_b200.so> <new libnig_b200.so>
"""
import re
import subprocess
import sys


def kernels(so):
    out = subprocess.check_output(["cuobjdump", "-sass", so], text=True)
    ks, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            ks[cur] = []
            continue
        if cur is None:
            continue
        s = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line)            # instruction addresses
        s = re.sub(r"/\* 0x[0-9a-f]+ \*/", "", s).strip()      # encodings
        if s and not s.startswith("//") and not s.startswith("."):
            ks[cur].append(s)
    return ks


def main():
    a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
    diff = [k for k in a if k in b and a[k] != b[k]]
    missing = [k for k in a if k not in b]
    new = [k for k in b if k not in a]
    print(f"kernels in the first build: {len(a)}; identical in the second: {len(a) - len(diff) - len(missing)}; "
          f"differing: {len(diff)}; missing: {len(missing)}; new in the second: {len(new)}")
    for k in diff + missing:
        print("  differs / missing:", k)
    for k in new:
        print("  new:", k)
    return 1 if diff or missing else 0


if __name__ == "__main__":
    sys.exit(main())
