"""Static per-phase SASS instruction count of k_analyse<R1, MG, SP> from the built library (no GPU needed): every instruction is
attributed to the OUTERMOST source line of its inline chain (nvdisasm -gi) and mapped to a phase through the `// ====`
section markers of fx_analyse.cu, as tools/ncu_phases.py does with executed counts.  Inner loops count once, so this is a
proxy for the executed instructions per frame -- good for comparing builds before spending GPU time.
Usage: sass_phases.py [R1=16] [MG=0] [lib] [SP=0]"""
import collections, os, re, subprocess, sys, tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R1 = int(sys.argv[1]) if len(sys.argv) > 1 else 16
MG = int(sys.argv[2]) if len(sys.argv) > 2 else 0
lib = sys.argv[3] if len(sys.argv) > 3 else os.path.join(ROOT, "feature-extractor_b200/lib/libfxb200.so")
SP = int(sys.argv[4]) if len(sys.argv) > 4 else 0
src = open(os.path.join(ROOT, "feature-extractor_b200/csrc/fx_analyse.cu")).read().split("\n")


def find(needle):
    for i, l in enumerate(src):
        if needle in l:
            return i + 1
    raise SystemExit(f"marker {needle!r} not found")


marks = [
    ("helpers / prologue", 1),
    ("frame head (mbarrier wait)", find("for (int f = f_begin; f < f_end; ++f)")),
    ("filter + window + RMS", find("one-pole filter + window -> work array")),
    ("FFT-alpha gather", find("FFT-alpha: z = x w + i onepole")),
    ("split + spectral pass 1", find("previous non-silent spectrum of this thread's bins")),
    ("combine + flatness events", find("every thread needs the magnitude sum")),
    ("FFT-beta gather", find("FFT-beta: z = x + i 2^k P")),
    ("flatness prefetch + hop prefetch", find("The flatness product's continuation (record stage, below) starts")),
    ("pitch (cnd scan, lag search)", find("pitch: cumulative normalised difference + lag search")),
    ("harmonic (peaks, inharmonicity)", find("The harmonic and sub-octave bins of f0")),
    ("record stage", find("the frame's record (what K1b needs), one part per warp")),
    ("chunk epilogue", find("---- chunk epilogue")),
    ("(end)", find("K1b: the scalar tail of both analyser bodies")),
]
with tempfile.TemporaryDirectory() as td:
    subprocess.run(["cuobjdump", "-xelf", "all", lib], cwd=td, check=True, stdout=subprocess.DEVNULL)
    cub = [f for f in os.listdir(td) if f.startswith("fx_analyse.") and f.endswith(".cubin")][0]
    sass = subprocess.run(["nvdisasm", "-gi", "-c", os.path.join(td, cub)], capture_output=True, text=True).stdout.split("\n")
want = f"k_analyseILi{R1}ELb{MG}ELb{SP}E"
inside, cur, counts, core = False, None, collections.Counter(), collections.Counter()
for l in sass:
    if l.startswith(".text."):
        inside = want in l
        continue
    if not inside:
        continue
    m = re.search(r'//## File "([^"]+)", line (\d+)(.*)', l)
    if m:
        chain = re.findall(r'"([^"]+)", line (\d+)', m.group(3))
        f, n = (chain[-1] if chain else (m.group(1), m.group(2)))
        cur = (os.path.basename(f), int(n))
        continue
    if re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+\S", l) and cur:
        if cur[0] == "fx_analyse.cu":
            ph = [name for name, ln in marks if ln <= cur[1]][-1]
            counts[ph] += 1
        else:
            core[cur[0]] += 1
tot = sum(counts.values()) + sum(core.values())
print(f"# static SASS instructions of k_analyse<{R1},{'true' if MG else 'false'},{'true' if SP else 'false'}> by phase ({tot} in all; fft_core is a separate function)")
for name, _ in marks[:-1]:
    print(f"{name:40s} {counts[name]:6d}")
for f, c in core.items():
    print(f"{'(' + f + ')':40s} {c:6d}")
