"""Static SASS of the block solver kernel per source region (dev tool, no GPU needed).

Usage: python scripts/block_sass_regions.py <lib.so | .cubin> [kernel-substring] [source.cu]

Each instruction counts at its OUTERMOST line in the kernel's source file (needs -lineinfo), so inlined helpers count where
the kernel calls them.  The regions are the kernel's own section markers ("// ===== pass =====", ...), found in the source
file, so the table follows the code when lines move; the source must be the one the library was built from.  The kernel
defaults to the lean instantiation with nine FK rows, leg_solve_block_kernel<1, false>."""
import re
import sys
from collections import Counter
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent))
import sass_cost as SC

ROOT = Path(__file__).resolve().parent.parent
LOC = re.compile(r'//## File "([^"]+)", line (\d+)(.*)')
INL = re.compile(r'inlined at "([^"]+)", line (\d+)')
INS = re.compile(r"\s+/\*([0-9a-f]{4,5})\*/\s+(.*?);")
# (region, marker that opens it); a region ends where the next one opens
MARKERS = [("pass", "// ================= pass"), ("accumulate", "// ================= accumulate"),
           ("verify", "// ================= verify"), ("commit", "// ================= commit"),
           ("replay", "// ================= replay"), ("after the blocks", "// ---- carry the angles")]


def instructions(txt, src_name):
    """-> [(outermost line in src_name or None, opcode)]"""
    out, line = [], None
    for l in txt.split("\n"):
        m = LOC.search(l)
        if m:
            chain = [(m.group(1), int(m.group(2)))] + [(f, int(n)) for f, n in INL.findall(m.group(3))]
            mine = [n for f, n in chain if f.endswith(src_name)]
            line = mine[-1] if mine else None
            continue
        m = INS.match(l)
        if m:
            t = re.sub(r"^@!?U?P\w+\s+", "", m.group(2).strip())
            out.append((line, t.split()[0].split(".")[0]))
    return out


def main():
    lib = sys.argv[1]
    kern = sys.argv[2] if len(sys.argv) > 2 else "leg_solve_block_kernelILi1ELb0E"
    src = Path(sys.argv[3]) if len(sys.argv) > 3 else ROOT / "sequential-inverse-kinematics_b200" / "csrc" / "seqik_solver.cu"
    lines = src.read_text().split("\n")
    starts = []
    for name, mark in MARKERS:
        n = next(k for k, l in enumerate(lines, 1) if mark in l)
        starts.append((n, name))

    def region(n):
        if n is None:
            return "outside the source file"
        name = "before the pass"
        for lo, nm in starts:
            if n >= lo:
                name = nm
        return name

    ins = instructions(SC.disasm(lib, kern, ("-gi",)), src.name)
    per = {}
    by_line = Counter()
    for n, op in ins:
        per.setdefault(region(n), Counter())[op] += 1
        by_line[n] += 1
    print(f"{kern}: {len(ins)} instructions")
    print(f"{'region':24s} {'lines':>11s} {'instr':>6s}  top opcodes")
    bounds = {nm: lo for lo, nm in starts}
    ends = {nm: (starts[k + 1][0] - 1 if k + 1 < len(starts) else None) for k, (lo, nm) in enumerate(starts)}
    for name in ["before the pass"] + [nm for nm, _ in MARKERS] + ["outside the source file"]:
        if name not in per:
            continue
        c = per[name]
        rng = f"{bounds[name]}-{ends[name] or ''}" if name in bounds else ""
        top = " ".join(f"{op}:{k}" for op, k in c.most_common(6))
        print(f"{name:24s} {rng:>11s} {sum(c.values()):6d}  {top}")
    lo, hi = bounds["pass"], bounds["accumulate"]
    print("heaviest lines of the pass:", ", ".join(f"{n}:{k}" for n, k in sorted(
        ((n, k) for n, k in by_line.items() if n is not None and lo <= n < hi), key=lambda x: -x[1])[:8]))


if __name__ == "__main__":
    main()
