"""Static SASS census of xpbd_step_kernel by source phase (no GPU needed).

Compiles csrc/nb2_xpbd.cu with the product library's flags (strict fp, -lineinfo, sm_100a), disassembles one instantiation with
`nvdisasm -gi` and charges every instruction to the kernel line it was inlined into (the outermost inlined-at line).  Kernel lines
are grouped into the phases of the substep, located by the section comments of the kernel body.  Per phase it counts the
instructions and the ones that make long dependency chains or break basic blocks: FP64 arithmetic (DFMA / DMUL / DADD), CALL
into out-of-line routines (division / sqrt slow paths, libm fallbacks), FCHK, BSSY and global loads (LDG).

    python scripts/xpbd_sass_census.py [--src DIR] [--lanes 16 --warps 14] [-D NAME ...]

`--src` points at another checkout's csrc/ to census it with the same script (before / after tables).  A static count is not a
measurement: it shows where code sits, not where time goes.
"""

from __future__ import annotations

import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from newton_b200 import build  # noqa: E402

COUNTED = ["DFMA", "DMUL", "DADD", "CALL", "FCHK", "BSSY", "BRA", "LDG"]
# (phase, comment that opens it): a phase runs from its anchor to the next one.  Lines before the first anchor and after the
# iteration loop are the once-per-substep work.
ANCHORS = [
    ("contact solve", "// ---- [iteration] solve_body_contact_positions"),
    ("contact apply", "// ---- [iteration] ordered per-body sum"),
    ("joint apply", "// ---- [iteration] solve_body_joints"),
    ("setup + joint_f + integrate + write-back", "// ---- State.body_parent_f"),
]
JOINT_CALL = "bool act = solve_joint("


def phase_of_line(src_lines: list[str]):
    starts = []
    for name, anchor in ANCHORS:
        hits = [i + 1 for i, s in enumerate(src_lines) if anchor in s]
        if len(hits) != 1:
            raise SystemExit(f"anchor {anchor!r} found {len(hits)} times in nb2_xpbd.cu")
        starts.append((hits[0], name))
    call = [i + 1 for i, s in enumerate(src_lines) if JOINT_CALL in s]
    if len(call) != 1:
        raise SystemExit(f"{JOINT_CALL!r} found {len(call)} times")

    def phase(line: int) -> str:
        if line == call[0]:
            return "joint solve (solve_joint)"
        name = "setup + joint_f + integrate + write-back"
        for start, n in starts:
            if line >= start:
                name = n
        return name

    return phase


def census(src_dir: str, lanes: int, warps: int, defines: list[str]):
    src = os.path.join(src_dir, "nb2_xpbd.cu")
    with tempfile.TemporaryDirectory() as tmp:
        cubin = os.path.join(tmp, "xpbd.cubin")
        flags = [f for f in build.NVCC_FLAGS if not f.startswith("-Xcompiler") and f not in ("-fPIC", "-O2")]
        cmd = [build._nvcc(), *flags, *build.STRICT_FLAGS, *[f"-D{d}" for d in defines], "-Xptxas", "-v", "-cubin", src, "-o", cubin]
        ptxas = subprocess.run(cmd, check=True, capture_output=True, text=True).stderr
        nvdisasm = os.path.join(os.path.dirname(build._nvcc()), "nvdisasm")
        sass = subprocess.run([nvdisasm, "-gi", cubin], check=True, capture_output=True, text=True).stdout
    mangled = f"_ZN3nb216xpbd_step_kernelILi{lanes}ELb0ELi{warps}E"
    m = re.search(rf"Function properties for {mangled}\S*\n(.*)\n.*Used (\d+) registers", ptxas)
    regs = f"{m.group(2)} registers, {m.group(1).strip()}" if m else "register report not found"
    phase = phase_of_line(open(src).read().splitlines())
    counts = collections.defaultdict(collections.Counter)
    in_kernel, where = False, None
    for line in sass.splitlines():
        if line.startswith(".text."):
            in_kernel, where = line.startswith(f".text.{mangled}"), None
            continue
        if not in_kernel:
            continue
        if line.startswith("$") and line.endswith(":"):  # subroutines (slow paths, fallbacks) follow the kernel body
            where = "out-of-line routines"
            continue
        if line.lstrip().startswith("//## File") and where != "out-of-line routines":
            f, ln = re.findall(r'File "([^"]+)", line (\d+)', line)[0] if "inlined at" not in line else \
                re.findall(r'"([^"]+)", line (\d+)', line)[-1]
            where = phase(int(ln)) if os.path.basename(f) == "nb2_xpbd.cu" else "other"
            continue
        ins = re.match(r"\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)", line)
        if ins and where is not None:
            op = ins.group(1)
            c = counts[where]
            c["SASS"] += 1
            if op in COUNTED:
                c[op] += 1
    return counts, regs


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--src", default=os.path.join(ROOT, "newton_b200", "csrc"))
    ap.add_argument("--lanes", type=int, default=16)
    ap.add_argument("--warps", type=int, default=14)
    ap.add_argument("-D", dest="defines", action="append", default=[])
    a = ap.parse_args()
    counts, regs = census(a.src, a.lanes, a.warps, a.defines)
    total = sum(c["SASS"] for c in counts.values())
    print(f"xpbd_step_kernel<{a.lanes},false,{a.warps}> strict fp, sm_100a: {regs}")
    print(f"{'phase':44s} {'SASS':>6s} {'share':>6s} " + " ".join(f"{k:>5s}" for k in COUNTED))
    order = ["joint solve (solve_joint)", "joint apply", "contact solve", "contact apply", "setup + joint_f + integrate + write-back",
             "out-of-line routines"]
    for p in order + sorted(set(counts) - set(order)):
        c = counts.get(p, collections.Counter())
        print(f"{p:44s} {c['SASS']:6d} {100.0 * c['SASS'] / max(total, 1):5.1f}% " + " ".join(f"{c[k]:5d}" for k in COUNTED))
    allc = sum(counts.values(), collections.Counter())
    print(f"{'total':44s} {total:6d} {100.0:5.1f}% " + " ".join(f"{allc[k]:5d}" for k in COUNTED))


if __name__ == "__main__":
    main()
