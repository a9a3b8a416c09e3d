"""SASS digest of the rotation loop of ransac_hyp_t_kernel (csrc/jacobi_thread.cuh, run_kernel4_thread): the ptxas resource line,
the length of the loop (the backward branch whose body holds the warp vote of the rotation loop), its instruction histogram and
how its instructions split over the source lines of jacobi_thread.cuh.  Compiled with the build's flags (build.py); no GPU needed.
    python tools/jacobi_sass_digest.py [--csrc DIR] [--label TEXT]
--csrc points at another copy of csrc/ (e.g. the parent commit's, from `git archive`) for a before/after comparison."""
import argparse, collections, os, re, subprocess, sys, tempfile
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, os.path.join(ROOT, "computervision_objectdetection_featurematching_b200"))
import build  # noqa: E402

KERNEL = "_ZN3cvg19ransac_hyp_t_kernelENS_10RansacWorkEii"
ap = argparse.ArgumentParser()
ap.add_argument("--csrc", default=build.CSRC)
ap.add_argument("--label", default="")
a = ap.parse_args()

with tempfile.TemporaryDirectory() as tmp:
    obj = os.path.join(tmp, "ransac.o")
    r = subprocess.run([build.nvcc()] + build.COMPILE_FLAGS + ["-Xptxas", "-v", "-c", "-o", obj, os.path.join(a.csrc, "ransac.cu")],
                       capture_output=True, text=True, check=True)
    subprocess.run(["cuobjdump", "-xelf", "all", obj], cwd=tmp, capture_output=True, check=True)
    cubin = [f for f in os.listdir(tmp) if f.endswith(".cubin")][0]
    sass = subprocess.run(["nvdisasm", "-g", "-c", os.path.join(tmp, cubin)], capture_output=True, text=True, check=True).stdout
sass = sass[sass.index(f"//--------------------- .text.{KERNEL} "):]
sass = sass[:sass.find("//---------------------", 1) % (len(sass) + 1)]

ptxas, cur = [], None
for line in r.stderr.splitlines():
    m = re.search(r"Compiling entry function '(\S+)'", line)
    if m:
        cur = m.group(1)
    elif cur == KERNEL and ("registers" in line or "spill" in line or "smem" in line):
        ptxas.append(line.split("ptxas info    :")[-1].strip())

# instructions in address order with their source line (nvdisasm -g prints `//## File "...", line N` before a run of them)
ins, src, label = [], None, {}
for line in sass.splitlines():
    m = re.search(r'//## File "([^"]+)", line (\d+)', line)
    if m:
        src = (os.path.basename(m.group(1)), int(m.group(2)))
        continue
    m = re.match(r"(\.L_x_\d+):", line.strip())
    if m:
        label[m.group(1)] = len(ins)                # index of the next instruction
        continue
    m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P[T\d]\s+)?([A-Z0-9_.]+)([^;]*);", line)
    if m:
        ins.append((int(m.group(1), 16), m.group(2), m.group(3), src))
loops = []
for i, (pc, op, args, _) in enumerate(ins):
    t = re.search(r"\((\.L_x_\d+)\)", args)
    if op.startswith("BRA") and t and label.get(t.group(1), i + 1) <= i:
        body = ins[label[t.group(1)]:i + 1]
        if any(x[1].startswith("VOTE") for x in body):
            loops.append(body)
body = min(loops, key=len)                      # the innermost loop holding the vote: the rotation loop
hist = collections.Counter(x[1].split(".")[0] for x in body)
lines = collections.Counter(x[3][1] for x in body if x[3] and x[3][0] == "jacobi_thread.cuh")
print(f"== ransac_hyp_t_kernel rotation loop {a.label}".rstrip())
for l in ptxas:
    print("   ptxas:", l)
print(f"   rotation loop: {len(body)} SASS instructions (0x{body[0][0]:x} .. 0x{body[-1][0]:x})")
print("   histogram:", ", ".join(f"{k} {v}" for k, v in hist.most_common()))
print("   by line of jacobi_thread.cuh (the compiler's attribution; inlined helpers count at their own lines):")
for ln, n in sorted(lines.items()):
    print(f"      {ln:4d}: {n}")
other = len(body) - sum(lines.values())
if other:
    print(f"      other files: {other}")
