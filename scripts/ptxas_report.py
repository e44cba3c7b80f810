"""Compile every translation unit of libsoftrod.so with -Xptxas -v (into a temporary directory; the library in the
tree is left alone) and print registers, stack and spills per kernel, one line each, sorted by kernel name."""
import concurrent.futures, os, re, subprocess, sys, tempfile
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gym_softrobot_b200 import build as b


def ptxas(tu, out_dir):
    name, src, defs, _ = tu
    cmd = [b._nvcc()] + b.NVCC_FLAGS + defs + ["-Xptxas", "-v", "-c", os.path.join(b.CSRC, src),
                                               "-o", os.path.join(out_dir, name + ".o")]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        sys.exit(f"nvcc failed on {name}:\n{res.stdout}")
    return res.stdout


with tempfile.TemporaryDirectory() as tmp, concurrent.futures.ThreadPoolExecutor(os.cpu_count() or 1) as ex:
    out = "\n".join(ex.map(lambda tu: ptxas(tu, tmp), b.translation_units()))
rows, cur, spill = {}, None, None
for line in out.splitlines():
    m = re.search(r"Compiling entry function '(\S+)'", line)
    if m:
        cur, spill = m.group(1), None
    m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
    if m and cur and spill is None:
        spill = m.groups()
    m = re.search(r"Used (\d+) registers", line)
    if m and cur:
        rows[cur] = (m.group(1),) + spill
        cur = None
names = subprocess.run(["c++filt"], input="\n".join(rows), stdout=subprocess.PIPE, text=True).stdout.splitlines()
MODELS = ["PLAIN", "PLANE", "MUSCLE", "ASSEMBLY", "FILTER", "SPLINE", "PLANAR"]   # LeanModel / LeanLayout (csrc/launch.cuh),
LAYOUTS = ["CTA", "FOLD", "CLUSTER"]                                            # in their order


def short(n):   # "void sr::k<..., (sr::LeanModel)2, (sr::LeanLayout)2>(args)" -> "k<..., MUSCLE, CLUSTER>"
    n = re.sub(r"\(sr::LeanModel\)(\d+)", lambda m: MODELS[int(m.group(1))], n)
    n = re.sub(r"\(sr::LeanLayout\)(\d+)", lambda m: LAYOUTS[int(m.group(1))], n)
    return re.sub(r"\(.*", "", n).replace("void sr::", "")


for name, (regs, stack, st, ld) in sorted(zip(map(short, names), rows.values())):
    print(f"{name:55s} regs={regs:>3s} stack={stack:>5s} spill_st={st:>5s} spill_ld={ld:>5s}")
