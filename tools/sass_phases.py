"""SASS footprint of each phase of the one-kernel flat step, for every instance of flat_step_kernel in the library.

Every phase of the step runs once per launch and the L2 flush between training steps evicts the kernel's code, so
the instruction bytes a phase walks through are a cost of their own.  This disassembles the library with
`nvdisasm --print-line-info-inline` (the library is built with -lineinfo), attributes each instruction to the line
of the kernel body it was inlined into, and groups the lines by the phase markers of csrc/fused_step.cuh
(`// ===... P<k>`, the final sums, the exit).  Runs on the CPU.

    python tools/sass_phases.py [library] [--source fused_step.cuh] [--json]

The library defaults to $CVCL_B200_LIB, else the in-tree build.  --source names the fused_step.cuh the library
was built from (default: the tree's), so that an older build can be read against its own line numbers.
"""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
from collections import OrderedDict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "multimodal-baby_b200", "csrc", "fused_step.cuh")
LIB = os.path.join(ROOT, "multimodal-baby_b200", "lib", "libcvcl_b200.so")
INSN_BYTES = 16                                  # every sm_100 instruction is 128 bits

LOC = re.compile(r'File "([^"]+)", line (\d+)')
INSN = re.compile(r"^\s+/\*[0-9a-f]+\*/\s+\S")


def phase_of_line(src_path):
    """line number -> phase label, from the phase markers of the kernel body"""
    marks = []
    with open(src_path) as fh:
        for i, line in enumerate(fh, 1):
            m = re.search(r"// =+ (P\d)", line)
            if m:
                marks.append((i, m.group(1)))
            elif "// ---- final sums" in line:
                marks.append((i, "final sums"))
            elif re.match(r"^done:", line):
                marks.append((i, "exit"))
            elif re.match(r"^flat_step_kernel\(", line):
                marks.append((i, "entry"))
    marks.sort()
    if not marks or marks[0][1] != "entry":
        raise SystemExit("no flat_step_kernel definition in %s" % src_path)

    def lookup(n):
        label = None
        for i, name in marks:
            if n >= i:
                label = name
        return label
    return lookup


def disassemble(lib, tmp):
    for tool in ("cuobjdump", "nvdisasm"):
        if not shutil.which(tool) and not os.path.exists("/usr/local/cuda/bin/" + tool):
            raise SystemExit("%s not found" % tool)
    exe = lambda t: shutil.which(t) or "/usr/local/cuda/bin/" + t
    subprocess.run([exe("cuobjdump"), "-xelf", "all", os.path.abspath(lib)], cwd=tmp, check=True,
                   capture_output=True)
    cubins = [f for f in os.listdir(tmp) if f.endswith(".cubin") and "sm_100" in f]
    if not cubins:
        raise SystemExit("no sm_100 cubin in %s" % lib)
    return subprocess.run([exe("nvdisasm"), "-gi", "-c", os.path.join(tmp, cubins[0])], check=True,
                          capture_output=True, text=True).stdout


def count(text, lookup, src_name):
    """{kernel symbol: OrderedDict(phase -> instructions)}"""
    out, cur, where = {}, None, None
    for line in text.splitlines():
        if line.startswith("//----") and ".text." in line:
            sym = line.split(".text.", 1)[1].split()[0]
            cur = OrderedDict() if "flat_step_kernel" in sym else None
            if cur is not None:
                out[sym] = cur
            where = None
            continue
        if cur is None:
            continue
        if "//##" in line:
            # the outermost location of the inlining chain is the line of the kernel body
            locs = LOC.findall(line)
            f, n = locs[-1]
            where = lookup(int(n)) if os.path.basename(f) == src_name else None
            continue
        if INSN.match(line):
            key = where or "out of line"
            cur[key] = cur.get(key, 0) + 1
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("lib", nargs="?", default=os.environ.get("CVCL_B200_LIB") or LIB)
    ap.add_argument("--source", default=SRC)
    ap.add_argument("--json", action="store_true")
    a = ap.parse_args()
    lookup = phase_of_line(a.source)
    tmp = tempfile.mkdtemp(prefix="sass_phases_")
    try:
        res = count(disassemble(a.lib, tmp), lookup, os.path.basename(a.source))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if not res:
        raise SystemExit("no flat_step_kernel in %s" % a.lib)
    if a.json:
        print(json.dumps({k: dict(v, total=sum(v.values())) for k, v in res.items()}))
        return
    order = ["entry", "P0", "P1", "P2", "P3", "P4", "P5", "final sums", "P6", "exit", "out of line"]
    for sym, ph in res.items():
        tot = sum(ph.values())
        print("%s  (%s)" % (sym, a.lib))
        for k in order + [k for k in ph if k not in order]:
            if k in ph:
                print("  %-12s %6d instructions  %7.1f KB" % (k, ph[k], ph[k] * INSN_BYTES / 1024))
        print("  %-12s %6d instructions  %7.1f KB" % ("total", tot, tot * INSN_BYTES / 1024))


if __name__ == "__main__":
    sys.exit(main())
