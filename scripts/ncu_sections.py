"""Executed warp-instructions and stall samples of one .cu file grouped by '// ----' section comments.
  python scripts/ncu_sections.py <report.ncu-rep> <file.cu>
"""
import csv, subprocess, sys, collections, re
rep, cu = sys.argv[1], sys.argv[2]
base = cu.split("/")[-1]
raw = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv", "--print-source", "cuda,sass"], capture_output=True, text=True).stdout
rows = list(csv.reader(raw.splitlines()))
lines = open(cu).read().splitlines()
marks = [(i + 1, l.strip()[:90]) for i, l in enumerate(lines)
         if re.match(r"\s*// ----", l) or re.match(r"^(NB2_DEV|NB2_CALL|__global__|static|template)\b.*\(", l)]
def section(ln):
    name = "(before first section)"
    for m, t in marks:
        if m <= ln: name = f"{m}: {t}"
        else: break
    return name
cur = hdr = None; seen = set(); inst = collections.Counter(); samp = collections.Counter()
for r in rows:
    if len(r) == 2 and r[0] == "File Path": cur = r[1].split("/")[-1]; continue
    if r and r[0] == "Line No": hdr = r; continue
    if hdr and len(r) == len(hdr) and r[2] == "-":
        try: n = int(r[hdr.index("Instructions Executed")]); s = int(r[hdr.index("# Samples")])
        except ValueError: continue
        key = (cur, r[0])
        if key in seen: continue
        seen.add(key)
        k = section(int(r[0])) if cur == base else "inlined helpers: " + cur
        inst[k] += n; samp[k] += s
ti, ts = sum(inst.values()), sum(samp.values())
print(f"# {rep}: {ti} warp-instructions, {ts} stall samples; grouped by section comments of {base}")
for k, v in sorted(inst.items(), key=lambda kv: -samp[kv[0]]):
    print(f"{v/ti*100:5.1f}% inst  {samp[k]/max(ts,1)*100:5.1f}% time(samples)  {k}")
