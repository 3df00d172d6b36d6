"""Check that two builds of the library carry the same kernels, instruction for instruction.

    python scripts/compare_sass.py <csrc dir A> <csrc dir B>

Each directory is a `make all` of mcp_raytracer_b200/csrc (libmcprt_b200.so, libmcprt_b200_count.so and their ptxas -v
logs build.log, build_count.log).  For both libraries it compares:
  - the set of functions in the `cuobjdump -sass` listing;
  - per function, every instruction and its `/* 0x... */` encoding words (which carry the scheduling control bits), with
    only the `/*0000*/` address comments removed;
  - per function, the ptxas registers, stack frame and spill lines.
Exit status 0 when everything is identical, 1 otherwise.  A host-only refactor of rt_api.cu must pass this.
"""
import re
import subprocess
import sys
from collections import Counter
from pathlib import Path

LIBS = (("libmcprt_b200.so", "build.log"), ("libmcprt_b200_count.so", "build_count.log"))
ADDR = re.compile(r"/\*[0-9a-f]{4,}\*/")


def sass(lib):
    """{(elf identifier, function): [instruction lines]} of `cuobjdump -sass lib`."""
    out = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True, check=True).stdout
    funcs, ident, cur = {}, "", None
    for line in out.splitlines():
        if line.startswith("Fatbin "):  # the next ELF's header (it may carry a "compressed" line): no function's code
            cur = None
        elif line.startswith("identifier = "):
            ident, cur = line[len("identifier = "):].strip(), None
        elif line.strip().startswith("Function : "):
            key = (ident, line.split("Function : ", 1)[1].strip())
            if key in funcs:
                raise SystemExit(f"{lib}: function listed twice: {key}")
            cur = funcs[key] = []
        elif cur is not None and line.strip():
            cur.append(ADDR.sub("", line).strip())
    return funcs


def ptxas(log):
    """Multiset of (function, stack/spill line, registers line) from a ptxas -v log."""
    lines = Path(log).read_text().splitlines()
    rows = []
    for i, line in enumerate(lines):
        m = re.search(r"Function properties for (\S+)", line)
        if not m:
            continue
        props = lines[i + 1].strip() if i + 1 < len(lines) else ""
        used = lines[i + 2].strip() if i + 2 < len(lines) and "Used" in lines[i + 2] else ""
        rows.append((m.group(1), props, re.sub(r"^ptxas info\s*:\s*", "", used)))
    return Counter(rows)


def main():
    if len(sys.argv) != 3:
        raise SystemExit(__doc__)
    a, b = Path(sys.argv[1]), Path(sys.argv[2])
    ok = True
    for lib, log in LIBS:
        fa, fb = sass(a / lib), sass(b / lib)
        if set(fa) != set(fb):
            ok = False
            for k in sorted(set(fa) - set(fb)):
                print(f"{lib}: only in A: {k[1]} ({k[0]})")
            for k in sorted(set(fb) - set(fa)):
                print(f"{lib}: only in B: {k[1]} ({k[0]})")
        differ = [k for k in sorted(set(fa) & set(fb)) if fa[k] != fb[k]]
        for k in differ:
            print(f"{lib}: SASS differs: {k[1]} ({k[0]})")
        ok &= not differ
        pa, pb = ptxas(a / log), ptxas(b / log)
        for row in sorted((pa - pb) + (pb - pa)):
            print(f"{log}: ptxas -v differs: {row}")
        ok &= pa == pb
        print(f"{lib}: {len(fa)} / {len(fb)} functions, {sum(map(len, fa.values()))} SASS lines in A, "
              f"{len(differ)} differ; {sum(pa.values())} ptxas property rows")
    print("IDENTICAL" if ok else "DIFFERENT")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
