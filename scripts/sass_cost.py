"""Static cost sheet of a kernel's SASS: per region (source-line ranges) instruction counts, branch counts and the
sum of the compiler's stall counts (the issue cycles one warp alone needs when no scoreboard wait fires).
Usage: python scripts/sass_cost.py <lib.so|cubin> <kernel-name-substring> [region=hexaddr ...]   (regions split the loop body
by address; SASS_COLD="file:lo-hi,..." marks source ranges as cold)
Reads `nvdisasm -g -hex` style output (line info needs -lineinfo).  A development aid: the numbers only rank variants
of the same kernel before spending GPU time."""
import re
import subprocess
import sys
import tempfile
from collections import defaultdict
from pathlib import Path


def disasm(path, kernel, flags=("-g", "-hex")):
    path = Path(path)
    tmp = Path(tempfile.mkdtemp())
    if path.suffix != ".cubin":
        subprocess.run(["cuobjdump", "-xelf", "all", str(path.resolve())], cwd=tmp, check=True, stdout=subprocess.DEVNULL)
        cubins = list(tmp.glob("*.cubin"))
    else:
        cubins = [path]
    for cb in cubins:
        txt = subprocess.run(["nvdisasm", *flags, str(cb)], capture_output=True, text=True).stdout
        m = re.search(r"^\.text\.(\S*%s\S*):" % re.escape(kernel), txt, re.M)
        if m:
            start = m.start()
            nxt = re.search(r"^\.text\.", txt[m.end():], re.M)
            return txt[start: m.end() + nxt.start() if nxt else len(txt)]
    raise SystemExit(f"kernel {kernel} not found")


def parse(txt):
    """-> list of dict(addr, op, text, line=(file, line), stall, wait, label)"""
    out = []
    cur = None
    pending = None
    for l in txt.split("\n"):
        m = re.search(r'//## File "([^"]+)", line (\d+)', l)
        if m:
            cur = (m.group(1).split("/")[-1], int(m.group(2)))
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,5})\*/\s+(.*?);\s*/\* (0x[0-9a-f]{16}) \*/", l)
        if m:
            pending = dict(addr=int(m.group(1), 16), text=m.group(2).strip(), line=cur, lo=int(m.group(3), 16))
            continue
        m = re.match(r"\s+/\* (0x[0-9a-f]{16}) \*/", l)
        if m and pending is not None:
            hi = int(m.group(1), 16)
            pending["stall"] = (hi >> 41) & 0xF
            pending["yield"] = (hi >> 45) & 1
            pending["wbar"] = (hi >> 46) & 7
            pending["rbar"] = (hi >> 49) & 7
            pending["wait"] = (hi >> 52) & 0x3F
            t = pending["text"]
            t = re.sub(r"^@!?U?P\d\s+", "", t)
            pending["op"] = t.split()[0].split(".")[0]
            out.append(pending)
            pending = None
            continue
        m = re.match(r"(\.L_x_\d+):", l)
        if m:
            out.append(dict(label=m.group(1)))
    return out


def sheet(ins, regions, cold):
    """regions: {name: predicate(line)}; cold: predicate(line) for blocks excluded from the hot sums."""
    rows = defaultdict(lambda: defaultdict(int))
    for i in ins:
        if "label" in i:
            continue
        ln = i["line"]
        for name, pred in regions.items():
            if pred(i):
                r = rows[name + (" (cold)" if cold(i) else "")]
                r["n"] += 1
                r["stall"] += max(i["stall"], 1)
                r["waits"] += 1 if i["wait"] else 0
                if i["op"] in ("BRA", "BSSY", "BSYNC", "CALL", "RET", "WARPSYNC"):
                    r["ctl"] += 1
                if i["op"] == "MUFU":
                    r["mufu"] += 1
                break
    return rows


if __name__ == "__main__":
    lib, kern = sys.argv[1], sys.argv[2]
    ins = parse(disasm(lib, kern))
    real = [i for i in ins if "label" not in i]
    print(f"{len(real)} instructions")
    # loop body of the pipe kernel: between the first VOTE.ANY (loop test) and the last
    votes = [k for k, i in enumerate(real) if i["text"].startswith("VOTE.ANY") or " VOTE.ANY" in i["text"]]
    lo, hi = (votes[0], votes[-1]) if len(votes) >= 2 else (0, len(real))
    body = real[lo:hi + 2]
    # split the body at the BSSY that opens the trip (the last top-level region): find by source line of `S.trip()` call
    # optional cold source ranges (rare paths excluded from the hot sums): SASS_COLD="seqik_core.cuh:100-127,seqik_core.cuh:540-590"
    import os
    cold_ranges = []
    for item in filter(None, os.environ.get("SASS_COLD", "").split(",")):
        f_, r_ = item.split(":")
        lo_, hi_ = r_.split("-")
        cold_ranges.append((f_, int(lo_), int(hi_)))

    def is_cold(i):
        f, n = i["line"] or ("", 0)
        return any(f.endswith(cf) and lo_ <= n <= hi_ for cf, lo_, hi_ in cold_ranges)
    # region boundaries: name=hexaddr ... (sorted); default: whole body
    marks = sorted((int(a.split("=")[1], 16), a.split("=")[0]) for a in sys.argv[3:])
    if not marks:
        marks = [(body[0]["addr"], "body")]
    def region_of(i):
        name = "pre"
        for addr, nm in marks:
            if i["addr"] >= addr:
                name = nm
        return name
    names = ["pre"] + [nm for _, nm in marks]
    regions = {nm: (lambda nm: lambda i: region_of(i) == nm)(nm) for nm in names}
    rows = sheet(body, regions, is_cold)
    print(f"loop body {body[0]['addr']:#x}..{body[-1]['addr']:#x}")
    for name in sorted(rows):
        r = rows[name]
        print(f"{name:18s} n={r['n']:5d} stall_sum={r['stall']:6d} ctl={r['ctl']:4d} mufu={r['mufu']:3d} sb_waits={r['waits']:4d}")
