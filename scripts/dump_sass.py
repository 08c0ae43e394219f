"""Writes profiles/sass/: full SASS of the two tcgen05 kernels and an opcode histogram per kernel
of liberp_b200.so (cuobjdump -sass).  Run after a build:  python scripts/dump_sass.py"""
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "erp_match_eightpoint_test_b200", "lib", "liberp_b200.so")
OUT = os.path.join(ROOT, "profiles", "sass")
os.makedirs(OUT, exist_ok=True)
txt = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
demangle = lambda n: subprocess.run(["c++filt", n], capture_output=True, text=True).stdout.strip()
kernels = collections.OrderedDict()
cur = None
for line in txt.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = m.group(1)
        kernels[cur] = []
        continue
    if cur and re.match(r"\s+/\*[0-9a-f]{4,}\*/", line):
        kernels[cur].append(re.sub(r"\s*/\* 0x[0-9a-f]+ \*/\s*$", "", line).rstrip())
FULL = {"knn2_tc_kernelILi2": "knn2_tc_kernel_D64.sass", "knn2_tc1_kernelILi1E": "knn2_tc1_kernel_D64.sass", "knn2_tc1_kernelILi2E": "knn2_tc1_kernel_D128.sass",
        "score_tc_kernel": "score_tc_kernel.sass", "min8_kernelILb0": "min8_kernel.sass", "refine_kernelILi2": "refine_kernel.sass",
        "score_list_kernel": "score_list_kernel.sass", "finish_kernelILi0": "finish_kernel.sass", "push_slots_kernel": "push_slots_kernel.sass",
        "xchg_best_kernel": "xchg_best_kernel.sass", "gather_slots_kernel": "gather_slots_kernel.sass", "argmax_plan_kernel": "argmax_plan_kernel.sass"}
with open(os.path.join(OUT, "opcode_histogram.txt"), "w") as f:
    f.write("# per kernel: instruction count and the opcodes that prove the Blackwell path\n"
            "# (UTC*MMA = tcgen05.mma, LDTM = tcgen05.ld, UTMALDG = TMA tensor load, UBLKCP = bulk copy, SYNCS = mbarrier)\n")
    for name, ins in kernels.items():
        ops = collections.Counter()
        for l in ins:
            m = re.search(r"\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", l)
            if m:
                ops[m.group(1).split(".")[0]] += 1
        key = {k: v for k, v in ops.items() if k.startswith(("UTC", "LDTM", "UTMA", "UBLKCP", "SYNCS", "DFMA", "DADD", "DMUL", "FFMA", "FSET", "REDUX", "ATOM", "HMMA"))}
        f.write(f"{demangle(name)[:110]}\n    {len(ins)} instructions; {dict(sorted(key.items()))}\n")
        for frag, fn in FULL.items():
            if frag in name:
                open(os.path.join(OUT, fn), "w").write(f"// {demangle(name)}\n" + "\n".join(ins) + "\n")
print("wrote", OUT)
