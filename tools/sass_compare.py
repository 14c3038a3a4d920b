"""Instruction-for-instruction comparison of k_analyse between two builds of fx_analyse.cu (no GPU needed): the parity-mode
instantiations of a build (third template argument false) against a build from before the spectrum mode existed, symbol names
ignored, and the static size of the power-mode instantiations.
Usage: sass_compare.py <old.cubin> <new.cubin>   (cubins from nvcc -cubin -gencode arch=compute_100a,code=sm_100a -O3 ...)"""
import re, subprocess, sys
def funcs(cubin):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout
    fs, cur = {}, None
    for l in out.split("\n"):
        m = re.match(r"\s+Function : (\S+)", l)
        if m: cur = m.group(1); fs[cur] = []; continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", l)
        if m and cur: fs[cur].append(re.sub(r"_Z\w+", "SYM", m.group(1)))
    return fs
a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
for R1 in (16, 8, 4):
    for MG in (0, 1):
        pa = [v for k, v in a.items() if f"k_analyseILi{R1}ELb{MG}EE" in k]
        pb = [v for k, v in b.items() if f"k_analyseILi{R1}ELb{MG}ELb0EE" in k]
        pp = [v for k, v in b.items() if f"k_analyseILi{R1}ELb{MG}ELb1EE" in k]
        assert len(pa) == 1 and len(pb) == 1 and len(pp) == 1
        print(f"k_analyse<{R1},{bool(MG)}>: parent {len(pa[0])} instr, Re^2 {len(pb[0])} instr, identical={pa[0] == pb[0]}; power {len(pp[0])} instr (+{len(pp[0]) - len(pa[0])})")
